"""GPU parity tests: the CUDA path (through the C ABI, via smvp_toolkit_b200.engine) against the oracle.

Bar (BASELINE.json north_star):  integer arrays bit-exact; y within 1e-12 relative L2 (fp64);
the deterministic TJDS variant bit-identical run to run.
"""
import math
import os

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle

pytestmark = pytest.mark.gpu

TOL = 1e-12  # relative L2, fp64 (north_star)


@pytest.fixture(scope="module")
def eng():
    import smvp_toolkit_b200 as e

    assert e.device_count() >= 1
    return e


def torch_view(arr):
    import torch

    return torch.as_tensor(arr, device="cuda")


def check_csr(eng, coo, m, n, x, variants=(1, 2)):
    rp, ci, va = oracle.csr_build(coo, m, n)
    A = eng.CsrMatrix.build(coo, m, n)
    g_rp, g_ci, g_va = A.export()
    assert np.array_equal(g_rp, rp), "row_ptr not bit-exact"
    assert np.array_equal(g_ci, ci), "col_ind not bit-exact"
    assert np.array_equal(g_va.view(np.int64), va.view(np.int64)), "val not bit-exact"
    y_ref = oracle.csr_mult(rp, ci, va, x)
    for v in variants:
        y, td = A.mult(x, iters=2, variant=v)
        assert util.rel_l2(y, y_ref) <= TOL, "variant %d" % v
        assert len(td.time_each) == 2 and td.time_total >= 0
        if np.linalg.norm(y_ref) == 0:
            assert np.all(y == 0)
    A.free()
    return y_ref


def check_tjds(eng, coo, m, n, x, y_csr):
    t = oracle.tjds_build(coo, m, n)
    A = eng.TjdsMatrix.build(coo, m, n)
    perm, sp, ri, va = A.export()
    assert A.ndiag == t.ndiag
    assert np.array_equal(perm, t.perm), "perm not bit-exact"
    assert np.array_equal(sp, t.start_pos), "start_pos not bit-exact"
    assert np.array_equal(ri, t.row_ind), "row_ind not bit-exact"
    assert np.array_equal(va.view(np.int64), t.val.view(np.int64)), "val not bit-exact"
    assert A.ref_diag_limit == t.ref_limit
    y_ref = oracle.tjds_mult(t, x)
    ya, _ = A.mult(x, iters=2, variant=eng.TJDS_ATOMIC)
    assert util.rel_l2(ya, y_ref) <= TOL
    assert util.rel_l2(ya, y_csr) <= TOL  # TJDS == CSR, pins x indexing
    for det in (eng.TJDS_DETERMINISTIC_FAST, eng.TJDS_DETERMINISTIC):  # one-word and two-word (exact) integer accumulation
        yd1, _ = A.mult(x, iters=1, variant=det)
        yd2, _ = A.mult(x, iters=3, variant=det)
        assert util.rel_l2(yd1, y_ref) <= TOL and util.rel_l2(yd1, y_csr) <= TOL
        assert np.array_equal(yd1.view(np.int64), yd2.view(np.int64)), "deterministic variant differs run to run"
    A.free()
    return yd1


# ---------------------------------------------------------------------------- sample matrices
@pytest.mark.parametrize("name", util.SAMPLES)
@pytest.mark.parametrize("xmode", ["ones", "random"])
def test_sample_matrices(eng, name, xmode):
    m, n, coo = util.load_sample(name)
    x = np.ones(n) if xmode == "ones" else np.random.default_rng(7).uniform(-1, 1, n)
    y_csr = check_csr(eng, coo, m, n, x)
    check_tjds(eng, coo, m, n, x, y_csr)


@pytest.mark.parametrize("name,alg", sorted(util.GOLDEN_REPORTS))
def test_golden_reports_through_reference_interface(eng, name, alg):
    """The reference's golden report files, through the mirrored entry points (x = ones)."""
    rep = util.parse_report(os.path.join(util.GOLDEN, "reports", util.GOLDEN_REPORTS[(name, alg)]))
    m, n, coo = util.load_sample(name)
    if alg == "CSR":
        y, td = eng.smvp_csr_compute(coo, m, len(coo), 3, fInputColumns=n)
    else:
        y, td = eng.smvp_tjds_compute(coo, m, n, len(coo), 3, ref_compat=True)  # the shipped truncation (U4/U5)
    assert len(td.time_each) == 3
    assert util.rel_l2(y, rep["y"]) <= 5e-6  # the files hold 6 significant digits
    # per element: 6 significant digits, with an absolute floor for rows that cancel to ~0 (memplus)
    scale = np.abs(coo["val"]).max() if len(coo) else 1.0
    assert np.all(np.abs(y - rep["y"]) <= 5e-6 * np.abs(rep["y"]) + 1e-12 * scale * 600)


# ---------------------------------------------------------------------------- random / edge cases
SHAPES = [
    (1, 1, 0), (1, 1, 1), (1, 7, 5), (7, 1, 4), (5, 5, 0), (17, 33, 100), (64, 64, 64 * 64), (300, 200, 3000),
    (1000, 1000, 20000), (2000, 50, 7000), (50, 2000, 7000), (4096, 4096, 50000), (10000, 10000, 10001),
]


@pytest.mark.parametrize("m,n,nnz", SHAPES)
@pytest.mark.parametrize("order", ["shuffled", "rowcol", "colrow"])
def test_random_matrices(eng, m, n, nnz, order):
    rng = np.random.default_rng(m * 1000003 + n * 101 + nnz)
    coo = util.random_coo(rng, m, n, nnz)
    if order == "rowcol":
        coo = coo[np.lexsort((coo["col"], coo["row"]))]
    elif order == "colrow":
        coo = coo[np.lexsort((coo["row"], coo["col"]))]
    x = rng.uniform(-3, 3, n)
    y_csr = check_csr(eng, coo, m, n, x)
    check_tjds(eng, coo, m, n, x, y_csr)


def test_skewed_rows_and_columns(eng):
    """One dense row, one dense column, many empty rows: the merge-path and segmented-TJDS cases."""
    rng = np.random.default_rng(99)
    m = n = 30000
    cells = set()
    for c in range(n):
        cells.add((123, c))
    for r in range(m):
        cells.add((r, 77))
    while len(cells) < 2 * n + 40000:
        r = int(rng.integers(0, m // 3)) * 3  # rows not divisible by 3 stay (mostly) empty
        cells.add((r, int(rng.integers(0, n))))
    rc = np.array(sorted(cells), dtype=np.int64)
    coo = oracle.make_coo(rc[:, 0], rc[:, 1], rng.uniform(-1, 1, len(rc)))
    rng.shuffle(coo)
    x = rng.uniform(-1, 1, n)
    y_csr = check_csr(eng, coo, m, n, x)
    check_tjds(eng, coo, m, n, x, y_csr)


def test_extreme_shapes(eng):
    """A row far longer than any tile (its partial crosses thousands of warp tiles and the fix-up chain), and a
    column far longer than a TJDS segment (one million jagged diagonals, tens of thousands of plan segments)."""
    rng = np.random.default_rng(31)
    # 3 x 2M, the middle row holds 1.5M entries
    n = 2_000_000
    c1 = np.sort(rng.choice(n, size=1_500_000, replace=False))
    rows = np.concatenate([np.zeros(5, np.int64), np.ones(len(c1), np.int64), np.full(7, 2)])
    cols = np.concatenate([np.arange(5) * 11, c1, np.arange(7) * 13 + 1])
    coo = oracle.make_coo(rows, cols, rng.uniform(-1, 1, len(rows)))
    rng.shuffle(coo)
    x = rng.uniform(-1, 1, n)
    y_csr = check_csr(eng, coo, 3, n, x)
    check_tjds(eng, coo, 3, n, x, y_csr)
    # 1M x 4, column 2 is dense (ndiag = 1M)
    m = 1_000_000
    rows = np.concatenate([np.arange(m), np.array([3, 999_999, 17])])
    cols = np.concatenate([np.full(m, 2), np.array([0, 0, 3])])
    coo = oracle.make_coo(rows, cols, rng.uniform(-1, 1, len(rows)))
    rng.shuffle(coo)
    x = rng.uniform(-1, 1, 4)
    y_csr = check_csr(eng, coo, m, 4, x)
    check_tjds(eng, coo, m, 4, x, y_csr)


def test_out_of_range_and_bad_args(eng):
    coo = oracle.make_coo([0, 5], [0, 1], [1.0, 2.0])
    with pytest.raises(eng.SmvpError) as ei:
        eng.CsrMatrix.build(coo, 3, 3)
    assert ei.value.code == eng.E_RANGE
    with pytest.raises(eng.SmvpError) as ei:
        eng.TjdsMatrix.build(coo, 3, 3)
    assert ei.value.code == eng.E_RANGE
    A = eng.CsrMatrix.build(oracle.make_coo([0], [0], [1.0]), 2, 2)
    with pytest.raises(eng.SmvpError) as ei:
        A.mult(np.ones(2), iters=0)
    assert ei.value.code == eng.E_ARG
    with pytest.raises(eng.SmvpError):
        A.mult(np.ones(2), iters=1, variant=9)


def test_time_stats_match_oracle(eng):
    ms = np.array([0.31, 0.29, 0.5, 0.30, 0.33])
    td = eng.TimeData(ms)
    s = oracle.time_stats(ms)
    assert (td.time_total, td.time_avg, td.time_min, td.time_max) == (s["total"], s["avg"], s["min"], s["max"])
    assert abs(td.time_stdev - s["stdev"]) <= 1e-15


# ---------------------------------------------------------------------------- synthetic generators
def test_stencil_generator_matches_numpy(eng):
    import torch

    nx, ny, nz = 5, 4, 3
    for (rb, re) in [(0, None), (7, 41)]:
        for mode in (0, 1):
            ref = synth_ref.stencil27(nx, ny, nz, rb, re, mode, seed=11)
            r, c, v = eng.synth_stencil27(nx, ny, nz, rb, re, mode, seed=11)
            assert r.n == len(ref)
            assert np.array_equal(torch_view(r).cpu().numpy(), ref["row"])
            assert np.array_equal(torch_view(c).cpu().numpy(), ref["col"])
            assert np.array_equal(torch_view(v).cpu().numpy(), ref["val"])
    counts = synth_ref.stencil27_row_counts(nx, ny, nz)
    pref = np.concatenate([[0], np.cumsum(counts)])
    for row in range(nx * ny * nz + 1):
        assert eng.synth_stencil27_prefix(nx, ny, nz, row) == pref[row]
    assert eng.synth_stencil27_prefix(369, 369, 369, 369 ** 3) == 1105 ** 3  # SURVEY.md 8: nnz of config 3


def test_rmat_generator_matches_numpy(eng):
    ref = synth_ref.rmat(10, 20000, seed=42)
    r, c, v = eng.synth_rmat(10, 20000, seed=42)
    assert r.n == len(ref)
    assert np.array_equal(torch_view(r).cpu().numpy(), ref["row"])
    assert np.array_equal(torch_view(c).cpu().numpy(), ref["col"])
    assert np.array_equal(torch_view(v).cpu().numpy(), ref["val"])


# ---------------------------------------------------------------------------- device-resident path, medium size
@pytest.mark.parametrize("kind", ["stencil", "rmat"])
def test_device_path_medium(eng, kind):
    """Device generators -> device builds -> device multiplies, against the oracle (seconds on the CPU)."""
    import torch

    if kind == "stencil":
        nx = 48
        m = n = nx ** 3
        r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=3)
    else:
        scale = 17
        m = n = 1 << scale
        r, c, v = eng.synth_rmat(scale, 16 << scale, seed=42)
    nnz = r.n
    coo = oracle.make_coo(torch_view(r).cpu().numpy(), torch_view(c).cpu().numpy(), torch_view(v).cpu().numpy())
    x = synth_ref.vector(n, 77)
    d_x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(d_x, n, 77)
    assert np.array_equal(d_x.cpu().numpy(), x)
    d_y = torch.empty(m, dtype=torch.float64, device="cuda")

    rp, ci, va = oracle.csr_build(coo, m, n)
    y_ref = oracle.csr_mult(rp, ci, va, x)
    A = eng.CsrMatrix.build_device(r, c, v, m, n, nnz)
    assert A.input_order == 1  # generators emit (row, col)-sorted lists
    g = A.export()
    assert np.array_equal(g[0], rp) and np.array_equal(g[1], ci) and np.array_equal(g[2], va)
    for variant in (eng.CSR_VECTOR, eng.CSR_MERGE, eng.CSR_AUTO):
        d_y.fill_(float("nan"))
        A.mult_device(d_x, d_y, variant)
        torch.cuda.synchronize()
        assert util.rel_l2(d_y.cpu().numpy(), y_ref) <= TOL, variant
    A.free()

    t = oracle.tjds_build(coo, m, n)
    T = eng.TjdsMatrix.build_device(r, c, v, m, n, nnz)
    perm, sp, ri, tv = T.export()
    assert np.array_equal(perm, t.perm) and np.array_equal(sp, t.start_pos)
    assert np.array_equal(ri, t.row_ind) and np.array_equal(tv, t.val)
    T.set_x_device(d_x)
    outs = []
    for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC):
        d_y.fill_(float("nan"))
        T.mult_device(d_y, variant)
        torch.cuda.synchronize()
        outs.append(d_y.cpu().numpy().copy())
        assert util.rel_l2(outs[-1], y_ref) <= TOL, variant
    assert np.array_equal(outs[1].view(np.int64), outs[2].view(np.int64))
    T.free()


@pytest.mark.parametrize("banded", [True, False])
def test_host_call_pipelined_transfers(eng, monkeypatch, banded):
    """smvp_csr_mult on a big matrix uploads x piece by piece under the first pass (a tile range starts once the
    leading part of x it reads has arrived) and copies y out range by range under the last pass.  Results must equal
    the plain copy-multiply-copy path bit for bit, for 1, 2 and 3 iterations, from pageable and from pinned host
    buffers, on a banded matrix (ranges really start early) and on one whose rows reach every column."""
    import ctypes

    import torch

    monkeypatch.setenv("SMVP_FORCE_OVERLAP", "1")  # numpy buffers are pageable: pipeline them anyway (slow but same path)
    m = n = (1 << 20) + 12345
    r = np.arange(m, dtype=np.int64)
    rows = [r, r[1:], r[:-1], r[3000:], r[:-3000]]
    cols = [r, r[1:] - 1, r[:-1] + 1, r[3000:] - 3000, r[:-3000] + 3000]
    if not banded:
        rows.append(r[::7])
        cols.append((r[::7] * 31 + 5) % n)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    key = np.unique(rows * n + cols)
    rng = np.random.default_rng(8)
    coo = oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))
    x = rng.uniform(-1, 1, n)
    y_ref = oracle.csr_mult(*oracle.csr_build(coo, m, n), x)
    A = eng.CsrMatrix.build(coo, m, n)
    outs = []
    for iters in (1, 2, 3):
        y, td = A.mult(x, iters=iters, variant=eng.CSR_MERGE)
        assert util.rel_l2(y, y_ref) <= TOL and len(td.time_each) == iters and td.time_min > 0
        outs.append(y)
    # pinned buffers straight through the C ABI, with a different x so that stale device data would show
    x2 = rng.uniform(-1, 1, n)
    hx = torch.as_tensor(x2).pin_memory()
    hy = torch.full((m,), float("nan"), dtype=torch.float64).pin_memory()
    rc = eng.lib().smvp_csr_mult(A._h, ctypes.c_void_p(hx.data_ptr()), ctypes.c_void_p(hy.data_ptr()), 1, None, eng.CSR_MERGE)
    assert rc == 0
    y_pinned = hy.numpy().copy()
    # pageable buffers without the force switch: served by plain copies, same bits
    monkeypatch.delenv("SMVP_FORCE_OVERLAP")
    y_pageable, _ = A.mult(x, iters=2, variant=eng.CSR_MERGE)
    assert np.array_equal(y_pageable.view(np.int64), outs[0].view(np.int64))
    monkeypatch.setenv("SMVP_NO_OVERLAP", "1")
    y_plain, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    y2_plain, _ = A.mult(x2, iters=1, variant=eng.CSR_MERGE)
    for y in outs:
        assert np.array_equal(y.view(np.int64), y_plain.view(np.int64))
    assert np.array_equal(y_pinned.view(np.int64), y2_plain.view(np.int64))
    A.free()


def test_host_call_pipelined_degenerate_shapes(eng, monkeypatch):
    """Shapes on which the pipelined host pass has little to pipeline: a tall matrix with 3 columns (x is one upload
    piece), a wide one with 4 rows (one tile range holds everything, the others are empty), a big matrix without a
    single nonzero (no range reads x), one whose FIRST row already reads the last column (every range waits
    for all of x), and one that reads only a window in the middle of x (the upload starts at the smallest column)."""
    monkeypatch.setenv("SMVP_FORCE_OVERLAP", "1")
    rng = np.random.default_rng(41)
    big = (1 << 21) + 777
    cases = []
    r = np.arange(big, dtype=np.int64)
    cases.append((big, 3, r, r % 3))                                              # tall
    c = np.sort(rng.choice(big, size=300000, replace=False))
    cases.append((4, big, rng.integers(0, 4, len(c)), c))                         # wide
    cases.append((big, big, np.zeros(0, np.int64), np.zeros(0, np.int64)))        # empty
    cases.append((big, big, np.concatenate([[0], r]), np.concatenate([[big - 1], np.maximum(r - 1, 0)])))  # first row reaches the end
    cases.append((big, 3 * big, r, big + 100 + (r * 7) % (big - 5000)))           # only a window of x is read (a GPU's row block)
    for m, n, rows, cols in cases:
        key = np.unique(np.asarray(rows, np.int64) * n + np.asarray(cols, np.int64))
        coo = oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))
        x = rng.uniform(-1, 1, n)
        y_ref = oracle.csr_mult(*oracle.csr_build(coo, m, n), x)
        A = eng.CsrMatrix.build(coo, m, n)
        for iters in (1, 2):
            y, td = A.mult(x, iters=iters, variant=eng.CSR_MERGE)
            assert util.rel_l2(y, y_ref) <= TOL, (m, n, iters)
            assert y.shape == (m,) and len(td.time_each) == iters
            if len(key) == 0:
                assert not y.any()
        A.free()


def _powerlaw_coo(rng, m, n, nnz, power):
    """Unique (row, col) pairs whose columns follow a power law spread over the whole index range (the hot columns
    are scattered by a multiplicative hash, as in an R-MAT matrix, not contiguous)."""
    rows = rng.integers(0, m, nnz)
    hot = np.minimum((n * rng.random(nnz) ** power).astype(np.int64), n - 1)
    cols = (hot * 2654435761) % n if math.gcd(2654435761, n) == 1 else hot
    key = np.unique(rows * n + cols)
    return oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))


def test_csr_relabel_forced_bit_identical(eng, monkeypatch):
    """The popularity relabelling of the column space (relabel.cu) is a multiply-side plan: the exported CSR
    arrays stay bit-exact against the oracle, and because entries keep their order inside each row, y is
    bit-identical with and without it -- for both kernels, through every entry point."""
    import torch

    rng = np.random.default_rng(77)
    m, n = 30011, 40009
    coo = _powerlaw_coo(rng, m, n, 600000, 4.0)
    x = rng.uniform(-1, 1, n)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y_ref = oracle.csr_mult(rp, ci, va, x)
    monkeypatch.setenv("SMVP_CSR_RELABEL", "0")
    P = eng.CsrMatrix.build(coo, m, n)
    plain = {v: P.mult(x, iters=1, variant=v)[0] for v in (eng.CSR_VECTOR, eng.CSR_MERGE)}
    assert P.x_relabel == -1
    monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
    A = eng.CsrMatrix.build(coo, m, n)
    for v in (eng.CSR_VECTOR, eng.CSR_MERGE):
        y, td = A.mult(x, iters=3, variant=v)
        assert A.x_relabel == 1
        assert util.rel_l2(y, y_ref) <= TOL
        assert np.array_equal(y.view(np.int64), plain[v].view(np.int64)), "relabelled y differs from the plain y"
    g = A.export()
    assert np.array_equal(g[0], rp) and np.array_equal(g[1], ci) and np.array_equal(g[2].view(np.int64), va.view(np.int64))
    # device entry points: explicit x, declared x (d_x = NULL), fan-out
    d_x = torch.as_tensor(x, device="cuda")
    d_y = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    for v in (eng.CSR_VECTOR, eng.CSR_MERGE):
        A.mult_device(d_x, d_y, v)
        torch.cuda.synchronize()
        assert np.array_equal(d_y.cpu().numpy().view(np.int64), plain[v].view(np.int64))
    x2 = rng.uniform(-1, 1, n)
    d_x2 = torch.as_tensor(x2, device="cuda")
    A.set_x_device(d_x2)
    P.set_x_device(d_x2)
    outs = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(2)]
    A.mult_device(None, outs[0], eng.CSR_MERGE)
    P.mult_device(None, outs[1], eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    assert util.rel_l2(outs[0].cpu().numpy(), oracle.csr_mult(rp, ci, va, x2)) <= TOL
    fan = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(2)]
    A.mult_device_fanout(None, [f.data_ptr() for f in fan], eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert torch.equal(fan[0], outs[0]) and torch.equal(fan[1], outs[0])
    # a handle that never saw set_x_device refuses d_x = NULL
    B = eng.CsrMatrix.build(coo, m, n)
    with pytest.raises(eng.SmvpError):
        B.mult_device(None, d_y, eng.CSR_MERGE)
    for h in (A, B, P):
        h.free()


def _hot_cold_coo(rng, m, n, nnz, hot_cols, hot_share):
    """Unique (row, col) pairs: `hot_share` of the entries fall on `hot_cols` columns scattered over the whole index
    range, the rest uniformly on all n columns."""
    rows = rng.integers(0, m, nnz)
    hot = (rng.integers(0, hot_cols, nnz) * 2654435761) % n
    cols = np.where(rng.random(nnz) < hot_share, hot, rng.integers(0, n, nnz))
    key = np.unique(rows * n + cols)
    return oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))


def test_csr_relabel_auto_decision(eng, monkeypatch):
    """AUTO relabels only when the handle touches at least MIN distinct columns AND the HOT most popular ones hold most
    of the nonzeros (>= 1/2 and >= 4x their fair share among the touched columns): a hot/cold matrix qualifies, a
    uniform one of the same shape does not; results stay within 1e-12 either way.  (MIN / HOT are 8 Mi / 4 Mi columns;
    the test scales them down through the tuning hooks.)  The big-matrix host path (pipelined copy-out, whole-x upload
    + permutation) is exercised on the way."""
    monkeypatch.setenv("SMVP_RELABEL_MIN_COLS", str(1 << 16))
    monkeypatch.setenv("SMVP_RELABEL_HOT_COLS", str(1 << 15))
    rng = np.random.default_rng(78)
    m, n, nnz = 200000, 2000003, 3000000
    x = rng.uniform(-1, 1, n)
    for hot_share, expect in ((0.7, 1), (0.0, -1)):
        coo = _hot_cold_coo(rng, m, n, nnz, 1 << 14, hot_share)
        rp, ci, va = oracle.csr_build(coo, m, n)
        y_ref = oracle.csr_mult(rp, ci, va, x)
        A = eng.CsrMatrix.build(coo, m, n)
        assert A.x_relabel == 0  # decided lazily, at the first pass
        for iters in (1, 2):
            y, _ = A.mult(x, iters=iters, variant=eng.CSR_MERGE)
            assert util.rel_l2(y, y_ref) <= TOL
        assert A.x_relabel == expect, (hot_share, A.x_relabel)
        g = A.export()
        assert np.array_equal(g[1], ci)
        A.free()


def test_csr_relabel_auto_keeps_banded_row_block(eng, monkeypatch):
    """Round-1 misfire (VERDICT r01, weak #1): the shard of one GPU out of 8 of a banded matrix reads a 1/8 window of
    x; measured against ALL columns that window looked like a hot set and the block was relabelled.  The decision is
    now taken over the columns the handle touches: a banded row block keeps its natural order (x_relabel == -1)
    whatever the size of the column space around it.  Thresholds scaled down as above: the block touches 60 002 of
    800 000 columns -- the old rule (fair share over all columns) relabelled exactly this shape."""
    import torch

    monkeypatch.setenv("SMVP_RELABEL_MIN_COLS", str(1 << 16))
    monkeypatch.setenv("SMVP_RELABEL_HOT_COLS", str(1 << 15))
    for m in (60000, 300000):  # below MIN touched columns; above it (then the hot set holds < 1/2 of a banded block)
        n, r0 = 800000, 350000
        rows = torch.arange(m, dtype=torch.int32, device="cuda").repeat_interleave(3)
        cols = ((rows + r0).view(-1, 3) + torch.tensor([-1, 0, 1], dtype=torch.int32, device="cuda")).reshape(-1).contiguous()
        vals = torch.tensor([-1.0, 26.0, -1.0], dtype=torch.float64, device="cuda").repeat(m)
        A = eng.CsrMatrix.build_device(rows, cols, vals, m, n, 3 * m)
        x = torch.ones(n, dtype=torch.float64, device="cuda")
        y = torch.empty(m, dtype=torch.float64, device="cuda")
        A.set_x_device(x)
        A.mult_device(None, y, eng.CSR_MERGE)
        torch.cuda.synchronize()
        assert A.x_relabel == -1, m
        assert bool((y == 24.0).all())
        A.free()


def test_tjds_relabel_forced(eng, monkeypatch):
    """Row-space relabelling of TJDS (the scatter side of the same plan): exported arrays unchanged, atomic variant
    within 1e-12, deterministic variant bit-identical to the natural-order handle, reference-compatible diagonal
    limit still honoured."""
    rng = np.random.default_rng(79)
    m, n = 40009, 30011
    coo_t = _powerlaw_coo(rng, n, m, 500000, 4.0)  # power law over the ROWS: build it transposed
    coo = oracle.make_coo(coo_t["col"], coo_t["row"], coo_t["val"])
    x = rng.uniform(-1, 1, n)
    t = oracle.tjds_build(coo, m, n)
    y_ref = oracle.csr_mult(*oracle.csr_build(coo, m, n), x)
    monkeypatch.setenv("SMVP_TJDS_RELABEL", "0")
    P = eng.TjdsMatrix.build(coo, m, n)
    y_det_plain, _ = P.mult(x, iters=1, variant=eng.TJDS_DETERMINISTIC)
    y_lim_plain, _ = P.mult(x, iters=1, variant=eng.TJDS_DETERMINISTIC, diag_limit=P.ref_diag_limit)
    assert P.y_relabel == -1
    monkeypatch.setenv("SMVP_TJDS_RELABEL", "1")
    A = eng.TjdsMatrix.build(coo, m, n)
    y_at, _ = A.mult(x, iters=2, variant=eng.TJDS_ATOMIC)
    assert A.y_relabel == 1
    assert util.rel_l2(y_at, y_ref) <= TOL
    y_det, _ = A.mult(x, iters=2, variant=eng.TJDS_DETERMINISTIC)
    assert util.rel_l2(y_det, y_ref) <= TOL
    assert np.array_equal(y_det.view(np.int64), y_det_plain.view(np.int64))
    y_lim, _ = A.mult(x, iters=1, variant=eng.TJDS_DETERMINISTIC, diag_limit=A.ref_diag_limit)
    assert np.array_equal(y_lim.view(np.int64), y_lim_plain.view(np.int64))
    perm, sp, ri, va = A.export()
    assert np.array_equal(perm, t.perm) and np.array_equal(sp, t.start_pos) and np.array_equal(ri, t.row_ind)
    A.free()
    P.free()


def test_fanout_and_write_only_y(eng):
    """smvp_csr_mult_device_fanout: one pass stores y into several destinations (the fused multi-GPU exchange writes
    peers' buffers this way); every destination must equal the plain result, for both kernels."""
    import torch

    rng = np.random.default_rng(12)
    m, n, nnz = 5000, 4000, 60000
    coo = util.random_coo(rng, m, n, nnz)
    x = rng.uniform(-1, 1, n)
    y_ref = oracle.csr_mult(*oracle.csr_build(coo, m, n), x)
    A = eng.CsrMatrix.build(coo, m, n)
    d_x = torch.as_tensor(x, device="cuda")
    for variant in (eng.CSR_VECTOR, eng.CSR_MERGE):
        outs = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3)]
        A.mult_device_fanout(d_x, [o.data_ptr() for o in outs], variant)
        torch.cuda.synchronize()
        for o in outs:
            assert util.rel_l2(o.cpu().numpy(), y_ref) <= TOL
        assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    with pytest.raises(eng.SmvpError):
        A.mult_device_fanout(d_x, [outs[0].data_ptr()] * 9, eng.CSR_MERGE)  # more than 8 destinations
    A.free()


def test_multi_gpu_operators_if_available(eng):
    """Row-block CSR (all exchanges) and column-block TJDS on 2 ranks, when the box has 2 GPUs."""
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (covered on CPU by tests/test_dist_gloo.py; run tools/check_multigpu.py on a multi-GPU box)")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29577", os.path.join(repo, "tools", "check_multigpu.py")],
                       capture_output=True, text=True, timeout=600)
    assert "MULTIGPU CHECK PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


# ---------------------------------------------------------------------------- BASELINE.json full size
def test_full_size_stencil_properties(eng):
    """Config 3 (27-point stencil 369^3, 1.35e9 nnz): size-independent properties, no oracle pass needed.
       (a) x = ones with the {26,-1} values: y_r = 27 - (entries in row r), exactly;
       (b) vector-CSR == merge-path CSR == TJDS(det) within 1e-12 on a random x;
       (c) linearity A(2 x1 - 3 x2) = 2 A x1 - 3 A x2 within 1e-12."""
    import torch

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = n = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    nnz = r.n
    assert nnz == (3 * nx - 2) ** 3
    A = eng.CsrMatrix.build_device(r, c, v, m, n, nnz)
    T = eng.TjdsMatrix.build_device(r, c, v, m, n, nnz)
    for a in (r, c, v):
        a.free()
    assert T.ndiag == 27
    counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda")
    expect = (27 - counts).to(torch.float64)
    row_ptr = torch.as_tensor(A.export_row_ptr()).to("cuda")
    assert torch.equal(row_ptr[1:] - row_ptr[:-1], counts.to(torch.int32))
    x1 = torch.ones(n, dtype=torch.float64, device="cuda")
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    for variant in (eng.CSR_VECTOR, eng.CSR_MERGE):
        y.fill_(float("nan"))
        A.mult_device(x1, y, variant)
        assert torch.equal(y, expect), variant
    T.set_x_device(x1)
    for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC):
        y.fill_(float("nan"))
        T.mult_device(y, variant)
        assert torch.equal(y, expect), variant

    xa = torch.empty(n, dtype=torch.float64, device="cuda")
    xb = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(xa, n, 1)
    eng.synth_vector(xb, n, 2)
    ya, yb, yc, yv = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(4))
    A.mult_device(xa, ya, eng.CSR_MERGE)
    A.mult_device(xb, yb, eng.CSR_MERGE)
    A.mult_device(2 * xa - 3 * xb, yc, eng.CSR_MERGE)
    lin = 2 * ya - 3 * yb
    assert float(torch.linalg.norm(yc - lin) / torch.linalg.norm(lin)) <= TOL
    A.mult_device(xa, yv, eng.CSR_VECTOR)
    assert float(torch.linalg.norm(yv - ya) / torch.linalg.norm(ya)) <= TOL
    T.set_x_device(xa)
    T.mult_device(yv, eng.TJDS_DETERMINISTIC)
    assert float(torch.linalg.norm(yv - ya) / torch.linalg.norm(ya)) <= TOL
    y2 = torch.empty_like(yv)
    T.mult_device(y2, eng.TJDS_DETERMINISTIC)
    assert torch.equal(y2, yv)
    A.free()
    T.free()


def test_full_size_rmat_scale26(eng, monkeypatch):
    """Configs 3/4 at FULL size (R-MAT scale 26, ~1.06e9 unique entries): where the popularity relabelling, the ranked
    cache hints, TJDS plans over 1e5+ jagged diagonals and the int32 edge cases actually engage (VERDICT r01, missing 6).
      (a) a 2^20-row slice and a 2^20-column slice of the matrix: CSR / TJDS arrays bit-exact against the oracle, the
          slice's rows of the full y within 1e-12 of the oracle's CSR loop (SURVEY.md 8d: "arrays bit-exact vs oracle on
          a <= 1 M-row slice");
      (b) the relabelled CSR multiply (AUTO picks it here) bit-identical to the natural-order one, merge vs vector
          within 1e-12;
      (c) TJDS atomic and deterministic within 1e-12 of CSR on the full matrix; deterministic bit-identical run to run.
    SMVP_TEST_RMAT_SCALE scales the test down for debugging."""
    import torch

    scale = int(os.environ.get("SMVP_TEST_RMAT_SCALE", "26"))
    m = n = 1 << scale
    r, c, v = eng.synth_rmat(scale, 16 << scale, seed=42)
    nnz = r.n
    d_x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(d_x, n, 4242)
    x = d_x.cpu().numpy()

    # ---- (b) full matrix, CSR: AUTO (relabelled at this size) and the natural order
    A = eng.CsrMatrix.build_device(r, c, v, m, n, nnz)
    y_auto = torch.empty(m, dtype=torch.float64, device="cuda")
    A.set_x_device(d_x)
    A.mult_device(None, y_auto, eng.CSR_MERGE)
    torch.cuda.synchronize()
    if scale >= 26:
        assert A.x_relabel == 1, "AUTO is expected to relabel the column space of R-MAT scale 26"
    y_vec = torch.empty_like(y_auto)
    A.mult_device(None, y_vec, eng.CSR_VECTOR)
    torch.cuda.synchronize()
    assert float(torch.linalg.norm(y_vec - y_auto) / torch.linalg.norm(y_auto)) <= TOL
    A.free()
    monkeypatch.setenv("SMVP_CSR_RELABEL", "0")
    P = eng.CsrMatrix.build_device(r, c, v, m, n, nnz)
    y_plain = torch.empty_like(y_auto)
    P.mult_device(d_x, y_plain, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert P.x_relabel == -1
    assert torch.equal(y_plain, y_auto), "relabelled and natural-order CSR must agree bit for bit"
    P.free()
    monkeypatch.delenv("SMVP_CSR_RELABEL")
    del y_vec, y_plain

    # ---- (c) full matrix, TJDS
    T = eng.TjdsMatrix.build_device(r, c, v, m, n, nnz)
    T.set_x_device(d_x)
    y_t = torch.empty(m, dtype=torch.float64, device="cuda")
    T.mult_device(y_t, eng.TJDS_ATOMIC)
    torch.cuda.synchronize()
    assert float(torch.linalg.norm(y_t - y_auto) / torch.linalg.norm(y_auto)) <= TOL
    T.mult_device(y_t, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    assert float(torch.linalg.norm(y_t - y_auto) / torch.linalg.norm(y_auto)) <= TOL
    y_t2 = torch.empty_like(y_t)
    T.mult_device(y_t2, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    assert torch.equal(y_t, y_t2), "deterministic TJDS differs run to run"
    assert T.ndiag > 1000
    T.free()
    del y_t, y_t2

    # ---- (a) slices against the oracle
    width = min(1 << 20, m // 4)
    y_host = y_auto.cpu().numpy()

    def pick(by_col):
        for start in (m // 2, 3 * (m // 4), m // 4 + m // 8, m // 8):
            if by_col:
                blk = eng.coo_filter_device(r, c, v, nnz, 0, m, start, start + width, 0, start)
            else:
                blk = eng.coo_filter_device(r, c, v, nnz, start, start + width, 0, n, start, 0)
            if 1000 <= blk[0].n <= 40_000_000:
                return start, blk
            for a in blk:
                a.free()
        raise AssertionError("no slice of a testable size")

    r0, (br, bc, bv) = pick(False)
    coo = oracle.make_coo(torch_view(br).cpu().numpy(), torch_view(bc).cpu().numpy(), torch_view(bv).cpu().numpy())
    rp, ci, va = oracle.csr_build(coo, width, n)
    S = eng.CsrMatrix.build_device(br, bc, bv, width, n, br.n)
    g = S.export()
    assert np.array_equal(g[0], rp) and np.array_equal(g[1], ci) and np.array_equal(g[2].view(np.int64), va.view(np.int64))
    S.free()
    y_ref = oracle.csr_mult(rp, ci, va, x)
    assert util.rel_l2(y_host[r0:r0 + width], y_ref) <= TOL
    for a in (br, bc, bv):
        a.free()

    c0, (br, bc, bv) = pick(True)
    coo = oracle.make_coo(torch_view(br).cpu().numpy(), torch_view(bc).cpu().numpy(), torch_view(bv).cpu().numpy())
    t = oracle.tjds_build(coo, m, width)
    S = eng.TjdsMatrix.build_device(br, bc, bv, m, width, br.n)
    perm, sp, ri, tv = S.export()
    assert S.ndiag == t.ndiag
    assert np.array_equal(perm, t.perm) and np.array_equal(sp, t.start_pos)
    assert np.array_equal(ri, t.row_ind) and np.array_equal(tv.view(np.int64), t.val.view(np.int64))
    S.free()
    for a in (br, bc, bv, r, c, v):
        a.free()


# ---------------------------------------------------------------------------- the batched `-n` loop (round 2)
@pytest.mark.parametrize("name", util.SAMPLES)
def test_batched_n_loop_matches_single_pass(eng, monkeypatch, name):
    """smvp_*_mult with many iterations on small matrices runs the loop batched (CUDA graphs; ONE looping CTA for the
    tiny sample files; the merge fix-up launched early): y must equal the single exact pass -- bit for bit for CSR and
    the deterministic TJDS variants, within 1e-12 for the atomic one -- for every variant, with batches that do and do
    not divide the iteration count, and the per-iteration times must be positive and complete."""
    m, n, coo = util.load_sample(name)
    x = np.random.default_rng(11).uniform(-1, 1, n)
    y_ref = oracle.csr_mult(*oracle.csr_build(coo, m, n), x)
    A = eng.CsrMatrix.build(coo, m, n)
    T = eng.TjdsMatrix.build(coo, m, n)
    for variant in (eng.CSR_AUTO, eng.CSR_VECTOR, eng.CSR_MERGE):
        y1, _ = A.mult(x, iters=1, variant=variant)
        for iters in (4, 50, 123):
            y, td = A.mult(x, iters=iters, variant=variant)
            assert util.rel_l2(y, y_ref) <= TOL
            if variant != eng.CSR_AUTO:  # AUTO may switch to the looping kernel (different lane layout, same tolerance)
                assert np.array_equal(y.view(np.int64), y1.view(np.int64)), (variant, iters)
            assert len(td.time_each) == iters and np.all(td.time_each > 0) and td.time_min > 0
    for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
        y1, _ = T.mult(x, iters=1, variant=variant)
        for iters in (4, 77):
            y, td = T.mult(x, iters=iters, variant=variant)
            assert util.rel_l2(y, y_ref) <= TOL
            if variant != eng.TJDS_ATOMIC:
                assert np.array_equal(y.view(np.int64), y1.view(np.int64)), (variant, iters)
            assert len(td.time_each) == iters and np.all(td.time_each > 0)
    # reference-compatible diagonal limit through the batched loop
    yl1, _ = T.mult(x, iters=1, variant=eng.TJDS_DETERMINISTIC, diag_limit=T.ref_diag_limit)
    yl, _ = T.mult(x, iters=40, variant=eng.TJDS_DETERMINISTIC, diag_limit=T.ref_diag_limit)
    assert np.array_equal(yl.view(np.int64), yl1.view(np.int64))
    # the switches that turn the batching off give the same vector
    monkeypatch.setenv("SMVP_EXACT_ITER_TIMES", "1")
    y, td = A.mult(x, iters=20, variant=eng.CSR_AUTO)
    assert util.rel_l2(y, y_ref) <= TOL and len(td.time_each) == 20
    monkeypatch.delenv("SMVP_EXACT_ITER_TIMES")
    monkeypatch.setenv("SMVP_NO_TINY_LOOP", "1")
    monkeypatch.setenv("SMVP_NO_PDL", "1")
    y, _ = A.mult(x, iters=20, variant=eng.CSR_AUTO)
    assert util.rel_l2(y, y_ref) <= TOL
    A.free()
    T.free()


def test_nonfinite_inputs_follow_ieee_propagation(eng):
    """ADVICE r01: the loader accepts 'inf' / 'nan' (strtod).  The exact integer accumulation needs finite input, so the
    deterministic variants route such a matrix or such an x to the atomic kernel (smvp_tjds_info_t.det_route == -1) and
    the affected rows come out Inf / NaN exactly as the CSR kernels and the reference's loop produce them; rows that
    the bad entries do not touch stay within 1e-12."""
    rng = np.random.default_rng(21)
    m, n, nnz = 3000, 2500, 40000
    coo = util.random_coo(rng, m, n, nnz)
    x = rng.uniform(-1, 1, n)

    def check(coo, x):
        rp, ci, va = oracle.csr_build(coo, m, n)
        with np.errstate(invalid="ignore", over="ignore"):
            y_ref = oracle.csr_mult(rp, ci, va, x)
        good = np.isfinite(y_ref)
        assert (~good).any() and good.any()
        A = eng.CsrMatrix.build(coo, m, n)
        yc, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
        A.free()
        T = eng.TjdsMatrix.build(coo, m, n)
        outs = [yc]
        for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
            y, _ = T.mult(x, iters=1, variant=variant)
            outs.append(y)
            if variant != eng.TJDS_ATOMIC:
                assert T.plan()[1] == -1, "non-finite input must be routed away from the integer kernel"
        T.free()
        for y in outs:
            assert np.array_equal(np.isnan(y), np.isnan(y_ref))
            assert np.array_equal(np.isposinf(y), np.isposinf(y_ref)) and np.array_equal(np.isneginf(y), np.isneginf(y_ref))
            assert util.rel_l2(y[good], y_ref[good]) <= TOL

    bad = coo.copy()
    bad["val"][17] = np.inf
    bad["val"][4321] = -np.inf
    bad["val"][999] = np.nan
    check(bad, x)                      # non-finite matrix entries
    xb = x.copy()
    xb[5] = np.inf
    xb[77] = np.nan
    check(coo, xb)                     # non-finite x
    # a finite x afterwards goes back to the integer kernel
    T = eng.TjdsMatrix.build(coo, m, n)
    T.mult(xb, iters=1, variant=eng.TJDS_DETERMINISTIC)
    assert T.plan()[1] == -1
    y, _ = T.mult(x, iters=1, variant=eng.TJDS_DETERMINISTIC)
    assert T.plan()[1] == 1
    assert util.rel_l2(y, oracle.csr_mult(*oracle.csr_build(coo, m, n), x)) <= TOL
    T.free()


def test_csr_relabel_forced_empty_rows_and_batched_loop(eng, monkeypatch):
    """A relabelled handle on a small power-law matrix with empty rows: y within 1e-12 of the oracle and bit-identical to
    a natural-order handle through the host entry point (iters 1 / 3 / 40; 40 takes the batched graph loop), the vector
    kernel, the device and the fan-out passes; the exported CSR arrays untouched."""
    import torch

    rng = np.random.default_rng(91)
    m, n = 50021, 40009
    coo = _powerlaw_coo(rng, m, n, 700000, 4.0)
    coo = coo[(coo["row"] % 97) != 5]  # some empty rows
    x = rng.uniform(-1, 1, n)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y_ref = oracle.csr_mult(rp, ci, va, x)

    def same(a, b):
        return np.array_equal(a.view(np.int64), b.view(np.int64))

    monkeypatch.setenv("SMVP_CSR_RELABEL", "0")
    B = eng.CsrMatrix.build(coo, m, n)
    y_nat, _ = B.mult(x, iters=1, variant=eng.CSR_MERGE)
    yv_nat, _ = B.mult(x, iters=1, variant=eng.CSR_VECTOR)
    assert B.x_relabel == -1
    B.free()
    monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
    A = eng.CsrMatrix.build(coo, m, n)
    for iters in (1, 3, 40):
        y, _ = A.mult(x, iters=iters, variant=eng.CSR_MERGE)
        assert util.rel_l2(y, y_ref) <= TOL, iters
        assert same(y, y_nat), iters
    assert A.x_relabel == 1
    yv, _ = A.mult(x, iters=1, variant=eng.CSR_VECTOR)
    assert util.rel_l2(yv, y_ref) <= TOL
    assert same(yv, yv_nat)
    g = A.export()
    assert np.array_equal(g[0], rp) and np.array_equal(g[1], ci) and np.array_equal(g[2].view(np.int64), va.view(np.int64))
    d_x = torch.as_tensor(x, device="cuda")
    d_y = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.set_x_device(d_x)
    A.mult_device(None, d_y, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert util.rel_l2(d_y.cpu().numpy(), y_ref) <= TOL
    assert same(d_y.cpu().numpy(), y_nat)
    outs = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(2)]
    A.mult_device_fanout(None, [o.data_ptr() for o in outs], eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert util.rel_l2(outs[0].cpu().numpy(), y_ref) <= TOL and torch.equal(outs[0], outs[1])
    assert same(outs[0].cpu().numpy(), y_nat)
    A.free()
