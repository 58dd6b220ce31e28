"""Row-pattern plan of CSR handles (pattern.cu, csr_pattern_kernel): which matrices take it, and that the kernel sums
every row in the reference loop's order -- y bit-identical to the oracle's sequential CSR loop."""
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


def _dump(*args):
    if not os.path.exists(LIB) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump not available")
    return subprocess.run([CUOBJDUMP, *args, LIB], capture_output=True, text=True, check=True).stdout


def test_pattern_kernel_spill_free_and_tma_staged():
    """Every instantiation of the pattern kernel keeps its registers (a spill halves the throughput of these kernels)
    and stages its tiles with TMA bulk copies."""
    res = _dump("-res-usage")
    names = re.findall(r"Function (\S*csr_pattern_kernel\S*):\s*\n\s*(REG:\d+ STACK:(\d+))", res)
    assert names, "no csr_pattern_kernel in the library"
    assert all(stack == "0" for _, _, stack in names), names
    for name, _, _ in names[:1]:
        assert "UBLKCP" in _dump("-sass", "-fun", name)


# ---------------------------------------------------------------------------- matrices
def _stencil27(nx, ny, nz, rng=None):
    coo = synth_ref.stencil27(nx, ny, nz)
    if rng is not None:
        coo["val"] = rng.uniform(-1, 1, len(coo))
    return nx * ny * nz, coo


def _from_lists(m, n, rows, cols, rng):
    rows, cols = np.concatenate(rows).astype(np.int64), np.concatenate(cols).astype(np.int64)
    key = np.unique(rows * n + cols)
    return oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))


def _stencil5_2d(nx, ny, rng):
    r = np.arange(nx * ny)
    ix, iy = r % nx, r // nx
    rows, cols = [r], [r]
    for dx, dy in ((-1, 0), (1, 0), (0, -1), (0, 1)):
        ok = (ix + dx >= 0) & (ix + dx < nx) & (iy + dy >= 0) & (iy + dy < ny)
        rows.append(r[ok])
        cols.append((ix + dx + nx * (iy + dy))[ok])
    return nx * ny, _from_lists(nx * ny, nx * ny, rows, cols, rng)


def _band(m, offsets, rng):
    r = np.arange(m)
    rows, cols = [], []
    for d in offsets:
        ok = (r + d >= 0) & (r + d < m)
        rows.append(r[ok])
        cols.append(r[ok] + d)
    return m, _from_lists(m, m, rows, cols, rng)


def _distinct_rows(npat, m, rng):
    """Rows 0 .. npat-2 hold {r, r + 1 + r}: one pattern each; every other row is the diagonal alone."""
    r = np.arange(m)
    k = np.arange(npat - 1)
    return m, _from_lists(m, m, [r, k], [r, 2 * k + 1], rng)


def _expected_patterns(coo, m, n):
    rp, ci, _ = oracle.csr_build(coo, m, n)
    lists = {tuple(ci[rp[r]:rp[r + 1]] - r) for r in range(m)}
    if max(len(t) for t in lists) > 32 or len(lists) > 256:
        return -1
    return len(lists)


def _cases():
    rng = np.random.default_rng(3)
    yield "stencil27 7x6x5", _stencil27(7, 6, 5, rng), 27
    yield "stencil27 33x3x35", _stencil27(33, 3, 35, rng), 27
    yield "stencil27 1x1x40", _stencil27(1, 1, 40, rng), 3
    yield "stencil27 2x1x50", _stencil27(2, 1, 50, rng), 6
    yield "stencil5 2-D 37x29", _stencil5_2d(37, 29, rng), 9
    yield "band 7", _band(5000, (-300, -2, -1, 0, 1, 2, 300), rng), None
    yield "band 32 wide", _band(3000, range(-16, 16), rng), None
    yield "band 33 wide", _band(3000, range(-16, 17), rng), -1
    yield "256 patterns", _distinct_rows(256, 2000, rng), 256
    yield "257 patterns", _distinct_rows(257, 2000, rng), -1
    m, n, nnz = 20000, 20000, 200000
    yield "random", (m, util.random_coo(rng, m, n, nnz)), -1


CASES = list(_cases())


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=[c[0] for c in CASES])
def test_row_patterns_decision_and_exact_rows(case):
    """AUTO takes the plan exactly when every row is one of at most 256 offset lists of at most 32 entries, numbers
    them, and the pattern kernel then reproduces the oracle's sequential loop bit for bit on random values and x."""
    import smvp_toolkit_b200 as eng

    name, (m, coo), expect = CASES[case]
    n = m
    want = _expected_patterns(coo, m, n)
    if expect is not None:
        assert want == expect, (name, want)
    rp, ci, va = oracle.csr_build(coo, m, n)
    x = np.random.default_rng(case).uniform(-1, 1, n)
    y_ref, _ = oracle.csr_mult_timed(rp, ci, va, x, 1)
    A = eng.CsrMatrix.build(coo, m, n)
    assert A.row_patterns == 0  # decided lazily, at the first pass
    y, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns == want, name
    if want > 0:
        assert np.array_equal(y.view(np.int64), y_ref.view(np.int64)), name
        info = eng.engine._CsrInfo()
        assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
        assert info.launches_per_mult[eng.CSR_MERGE] == 1  # no fix-up launch
    assert util.rel_l2(y, y_ref) <= TOL
    A.free()


@pytest.mark.gpu
def test_one_extra_entry_adds_one_pattern(monkeypatch):
    """A stencil with one more entry in one interior row has one more pattern; that row comes out right, and the
    merge kernel (plan forced off) agrees within 1e-12."""
    import smvp_toolkit_b200 as eng

    nx = 9
    m, coo = _stencil27(nx, nx, nx)
    r = 4 + nx * (4 + nx * 4)
    extra = oracle.make_coo(np.array([r]), np.array([r + 3 * nx]), np.array([0.5]))
    coo = np.concatenate([coo, extra])
    rng = np.random.default_rng(5)
    coo["val"] = rng.uniform(-1, 1, len(coo))
    x = rng.uniform(-1, 1, m)
    rp, ci, va = oracle.csr_build(coo, m, m)
    y_ref, _ = oracle.csr_mult_timed(rp, ci, va, x, 1)
    A = eng.CsrMatrix.build(coo, m, m)
    y, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns == 28
    assert np.array_equal(y.view(np.int64), y_ref.view(np.int64))
    monkeypatch.setenv("SMVP_CSR_PATTERN", "0")
    B = eng.CsrMatrix.build(coo, m, m)
    yb, _ = B.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert B.row_patterns == -1
    assert util.rel_l2(yb, y) <= TOL
    A.free()
    B.free()


@pytest.mark.gpu
def test_rmat_rejects_the_plan():
    import smvp_toolkit_b200 as eng

    r, c, v = eng.synth_rmat(14, 16 << 14)
    A = eng.CsrMatrix.build_device(r, c, v, 1 << 14, 1 << 14, r.n)
    for a in (r, c, v):
        a.free()
    x = np.random.default_rng(0).uniform(-1, 1, 1 << 14)
    A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns == -1
    A.free()


@pytest.mark.gpu
def test_device_pass_fanout_pipelined_host_call_and_batched_loop(monkeypatch):
    """On a stencil large enough for the pipelined host call (row ranges of the pattern kernel, x uploaded and y
    downloaded under the pass): host call == device pass == every fan-out destination, bit for bit, and the batched
    `-n` loop of a small stencil equals its single pass."""
    import torch

    import smvp_toolkit_b200 as eng

    monkeypatch.setenv("SMVP_FORCE_OVERLAP", "1")
    nx = 104  # rows + cols >= 2^21: the host call pipelines
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=7)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    dx = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(dx, m, 3)
    dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_device(dx, dy, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert A.row_patterns == 27
    outs = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3)]
    A.mult_device_fanout(dx, [o.data_ptr() for o in outs], eng.CSR_MERGE)
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o, dy)
    for iters in (1, 2):
        y, _ = A.mult(dx.cpu().numpy(), iters=iters, variant=eng.CSR_MERGE)
        assert np.array_equal(y.view(np.int64), dy.cpu().numpy().view(np.int64)), iters
    # against the merge kernel on the same handle data (plan forced off)
    monkeypatch.setenv("SMVP_CSR_PATTERN", "0")
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=7)
    B = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    ym = torch.empty_like(dy)
    B.mult_device(dx, ym, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert B.row_patterns == -1
    assert float(torch.linalg.norm(ym - dy) / torch.linalg.norm(dy)) <= TOL
    A.free()
    B.free()
    monkeypatch.delenv("SMVP_CSR_PATTERN")
    monkeypatch.delenv("SMVP_FORCE_OVERLAP")

    m, coo = _stencil27(12, 12, 12, np.random.default_rng(9))
    x = np.random.default_rng(10).uniform(-1, 1, m)
    S = eng.CsrMatrix.build(coo, m, m)
    y1, _ = S.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert S.row_patterns == 27
    for iters in (4, 50, 123):
        y, td = S.mult(x, iters=iters, variant=eng.CSR_MERGE)
        assert np.array_equal(y.view(np.int64), y1.view(np.int64)), iters
        assert len(td.time_each) == iters and np.all(td.time_each > 0)
    S.free()


@pytest.mark.gpu
def test_full_size_stencil_takes_the_plan():
    """369^3 (the benchmark's matrix): 27 patterns, x = ones gives the closed form 27 - (entries in the row) exactly,
    and a random x agrees with the vector kernel within 1e-12."""
    import torch

    import smvp_toolkit_b200 as eng

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda")
    x1 = torch.ones(m, dtype=torch.float64, device="cuda")
    y = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_device(x1, y, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert A.row_patterns == 27
    assert torch.equal(y, (27 - counts).to(torch.float64))
    xa = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(xa, m, 1)
    yv = torch.empty_like(y)
    A.mult_device(xa, y, eng.CSR_MERGE)
    A.mult_device(xa, yv, eng.CSR_VECTOR)
    assert float(torch.linalg.norm(yv - y) / torch.linalg.norm(y)) <= TOL
    A.free()
