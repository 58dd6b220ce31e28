"""Value width of the CSR row-pattern plan (pattern.cu, csr_pattern_kernel): the kernel streams fp16 or fp32 copies of
the values when every value converts to that type and back with the same 64 bits, and y stays bit-identical to the
oracle's sequential CSR loop at every width."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle
from test_dot import PAIRS, bits, reduce_partials, unit_partials

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(REPO, "smvp-toolkit_b200", "lib", "libsmvp_cuda.so")
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def _dump(*args):
    if not os.path.exists(LIB) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump not available")
    return subprocess.run([CUOBJDUMP, *args, LIB], capture_output=True, text=True, check=True).stdout


def test_pattern_kernels_at_every_width_widen_with_one_instruction():
    """Every pattern kernel exists at fp32 and fp16 (plain, epilogue, fan-out, dot), none spills, each stages with TMA
    and widens its values with F2F."""
    res = _dump("-res-usage")
    found = re.findall(r"Function (\S*csr_pattern_kernelI([dft])\S*):\s*\n\s*REG:\d+ STACK:(\d+)", res)
    by_type = {t: [n for n, tt, _ in found if tt == t] for t in ("d", "f", "t")}  # d: fp64, f: fp32, t: fp16 (uint16_t)
    assert all(len(v) == 4 for v in by_type.values()), {t: len(v) for t, v in by_type.items()}
    assert all(stack == "0" for _, _, stack in found), found
    for t, cvt in (("f", "F2F.F64.F32"), ("t", "F2F.F64.F16")):
        for name in by_type[t]:
            sass = _dump("-sass", "-fun", name)
            assert "UBLKCP" in sass and cvt in sass, name


# ---------------------------------------------------------------------------- matrices
def _csr_info(eng, A):
    info = eng.engine._CsrInfo()
    assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
    return info


def _structure(kind):
    """COO of a stencil-like matrix (values to be set)"""
    if kind == "stencil27":
        return 7 * 6 * 5, synth_ref.stencil27(7, 6, 5)
    if kind == "stencil27 b":
        return 33 * 3 * 35, synth_ref.stencil27(33, 3, 35)
    r = np.arange(37 * 29) if kind == "stencil5 2-D" else np.arange(5000)
    if kind == "stencil5 2-D":
        nx, ny = 37, 29
        ix, iy = r % nx, r // nx
        rows, cols = [r], [r]
        for dx, dy in ((-1, 0), (1, 0), (0, -1), (0, 1)):
            ok = (ix + dx >= 0) & (ix + dx < nx) & (iy + dy >= 0) & (iy + dy < ny)
            rows.append(r[ok])
            cols.append((ix + dx + nx * (iy + dy))[ok])
    else:  # band
        rows, cols = [], []
        for d in (-300, -2, -1, 0, 1, 2, 300):
            ok = (r + d >= 0) & (r + d < len(r))
            rows.append(r[ok])
            cols.append(r[ok] + d)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    key = np.unique(rows.astype(np.int64) * len(r) + cols)
    return len(r), oracle.make_coo(key // len(r), key % len(r), np.zeros(len(key)))


def _values(width, nnz, rng):
    """values that land on `width`: small integers (fp16), fp32-rounded uniforms (fp32), fp64 uniforms"""
    if width == 2:
        return rng.integers(-9, 10, nnz).astype(np.float64)
    v = rng.uniform(-1, 1, nnz)
    return v.astype(np.float32).astype(np.float64) if width == 4 else v


# (name, values, expected width); the values are tiled over the entries of a 7x6x5 27-point stencil
DECISIONS = [
    ("stencil {26, -1}", None, 2),
    ("all ones (pattern file)", [1.0], 2),
    ("65504 and 2^-24", [65504.0, 2.0 ** -24, -3.0], 2),
    ("-0.0 entries", [-0.0, 1.0, -0.0, 2.0], 2),
    ("2049", [2049.0, 1.0], 4),
    ("65520", [65520.0, 1.0], 4),
    ("1/3 rounded to fp32", [float(np.float32(1 / 3)), 1.0], 4),
    ("0.1", [0.1, 1.0], 8),
    ("fp64 subnormal", [5e-324, 1.0], 8),
    ("0.1 in the last row only", "last", 8),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(DECISIONS)), ids=[d[0] for d in DECISIONS])
def test_width_decision_and_exact_rows(case):
    """The narrowest width that holds every value bit for bit; 0 until the first pass; y bit-identical to the oracle."""
    import smvp_toolkit_b200 as eng

    name, vals, want = DECISIONS[case]
    m = 7 * 6 * 5
    coo = synth_ref.stencil27(7, 6, 5)
    if vals == "last":
        coo["val"] = 1.0
        coo["val"][-1] = 0.1
    elif vals is not None:
        coo["val"] = np.resize(np.array(vals, np.float64), len(coo))
    rp, ci, va = oracle.csr_build(coo, m, m)
    x = np.random.default_rng(case).uniform(-1, 1, m)
    y_ref, _ = oracle.csr_mult_timed(rp, ci, va, x, 1)
    A = eng.CsrMatrix.build(coo, m, m)
    assert _csr_info(eng, A).value_bytes == 0  # decided with the plan, at the first pass
    base = _csr_info(eng, A).device_bytes
    y, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns == 27 and A.value_bytes == want, (name, A.value_bytes)
    assert np.array_equal(y.view(np.int64), y_ref.view(np.int64)), name
    grown = _csr_info(eng, A).device_bytes - base
    assert grown == m + 4 * 27 * 33 + (want * len(coo) if want < 8 else 0), name  # pattern table + the narrow copy
    A.free()


@pytest.mark.gpu
def test_rejected_plan_has_no_width():
    """A matrix without the plan reports no width and holds no narrow copy."""
    import smvp_toolkit_b200 as eng

    m = 2000
    coo = util.random_coo(np.random.default_rng(0), m, m, 20000)  # far more than 256 offset lists
    coo["val"] = 1.0
    A = eng.CsrMatrix.build(coo, m, m)
    base = _csr_info(eng, A).device_bytes
    A.mult(np.ones(m), iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns == -1 and A.value_bytes == 0
    assert _csr_info(eng, A).device_bytes == base
    A.free()


MATRICES = ["stencil27", "stencil27 b", "stencil5 2-D", "band"]


@pytest.mark.gpu
@pytest.mark.parametrize("width", [2, 4, 8])
@pytest.mark.parametrize("kind", MATRICES)
def test_every_width_is_bit_identical(kind, width):
    """Plain pass == the oracle's loop; *_axpby == fl(alpha s) + fl(beta y0) on it; *_axpby_dot stores the same y and its
    dot equals the numpy restatement of the documented order (tiles of 32 rows, then dot_reduce's tree)."""
    import torch

    import smvp_toolkit_b200 as eng

    rng = np.random.default_rng(10 * MATRICES.index(kind) + width)
    m, coo = _structure(kind)
    coo["val"] = _values(width, len(coo), rng)
    rp, ci, va = oracle.csr_build(coo, m, m)
    x = rng.uniform(-1, 1, m)
    s_ref, _ = oracle.csr_mult_timed(rp, ci, va, x, 1)
    A = eng.CsrMatrix.build(coo, m, m)
    y, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.row_patterns > 0 and A.value_bytes == width
    assert np.array_equal(bits(y), bits(s_ref))
    dx = torch.as_tensor(x, device="cuda")
    w = rng.uniform(-1, 1, m)
    for alpha, beta in PAIRS:
        y0 = np.full(m, np.nan) if beta == 0.0 else rng.uniform(-2, 2, m)
        want = alpha * s_ref if beta == 0.0 else alpha * s_ref + beta * y0
        dy = torch.as_tensor(y0.copy(), device="cuda")
        A.mult_device_axpby(alpha, dx, beta, dy, eng.CSR_MERGE)
        assert np.array_equal(bits(dy.cpu().numpy()), bits(want)), (alpha, beta)
        for wv in (None, w):
            dy = torch.as_tensor(y0.copy(), device="cuda")
            dd = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
            A.mult_device_axpby_dot(alpha, dx, beta, dy, None if wv is None else torch.as_tensor(wv, device="cuda"), dd,
                                    eng.CSR_MERGE)
            assert np.array_equal(bits(dy.cpu().numpy()), bits(want)), (alpha, beta)
            dot = reduce_partials(unit_partials((want if wv is None else wv) * want, 32))
            assert bits(dd.cpu().numpy())[0] == bits(np.array([dot]))[0], (alpha, beta, wv is None)
    A.free()


@pytest.mark.gpu
@pytest.mark.parametrize("width", [2, 4])
def test_narrow_fanout_pipelined_host_call_and_batched_loop(monkeypatch, width):
    """A stencil large enough for the pipelined host call (row ranges of the pattern kernel), at a narrow width: device
    pass == the oracle's loop == every fan-out destination == the host call, bit for bit, and the batched `-n` loop of a
    small stencil equals its single pass."""
    import torch

    import smvp_toolkit_b200 as eng

    monkeypatch.setenv("SMVP_FORCE_OVERLAP", "1")
    nx = 104  # rows + cols >= 2^21: the host call pipelines
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    if width == 4:
        torch.as_tensor(v, device="cuda").mul_(1.0 + 2.0 ** -20)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    dx = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(dx, m, 3)
    dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_device(dx, dy, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert A.row_patterns == 27 and A.value_bytes == width
    rp, ci, va = A.export()
    x = dx.cpu().numpy()
    y_ref, _ = oracle.csr_mult_timed(rp, ci, va, x, 1)
    assert np.array_equal(bits(dy.cpu().numpy()), bits(y_ref))
    outs = [torch.full((m,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3)]
    A.mult_device_fanout(dx, [o.data_ptr() for o in outs], eng.CSR_MERGE)
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o, dy)
    for iters in (1, 2):
        y, _ = A.mult(x, iters=iters, variant=eng.CSR_MERGE)
        assert np.array_equal(bits(y), bits(y_ref)), iters
    A.free()
    monkeypatch.delenv("SMVP_FORCE_OVERLAP")

    m = 12 ** 3
    coo = synth_ref.stencil27(12, 12, 12)
    coo["val"] = _values(width, len(coo), np.random.default_rng(9))
    x = np.random.default_rng(10).uniform(-1, 1, m)
    S = eng.CsrMatrix.build(coo, m, m)
    y1, _ = S.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert S.row_patterns == 27 and S.value_bytes == width
    for iters in (4, 50, 123):
        y, _ = S.mult(x, iters=iters, variant=eng.CSR_MERGE)
        assert np.array_equal(bits(y), bits(y1)), iters
    S.free()


@pytest.mark.gpu
def test_full_size_stencil_streams_fp16():
    """369^3 (the benchmark's matrix, values {26, -1}): the plan streams fp16 values, and x = ones still gives the
    closed form 27 - (entries in the row) exactly."""
    import torch

    import smvp_toolkit_b200 as eng

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    x1 = torch.ones(m, dtype=torch.float64, device="cuda")
    y = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_device(x1, y, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert A.row_patterns == 27 and A.value_bytes == 2
    counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda")
    assert torch.equal(y, (27 - counts).to(torch.float64))
    A.free()
