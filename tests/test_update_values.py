"""In-place value update of CSR and TJDS handles (smvp_csr_update_values*, smvp_tjds_update_values*): after an update
the handle behaves exactly like a fresh build of the updated matrix once both have decided the same plans -- the same
exported arrays, the same info, the same y bits from every pass (TJDS atomic within 1e-12) -- while the structural plans
and the declared x stay, and every rejected list leaves the handle untouched."""
import ctypes
import os

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle
from test_tjds_exact import det_kernel_fast_flags

TOL = 1e-12
PAIRS = [(1.0, 0.0), (-1.0, 1.0), (2.5, -0.75)]
CSR_VARIANTS = (0, 1, 2)   # SMVP_CSR_AUTO, _VECTOR, _MERGE
TJDS_VARIANTS = (0, 1, 2)  # SMVP_TJDS_ATOMIC, _DETERMINISTIC, _DETERMINISTIC_FAST


@pytest.fixture(scope="module")
def eng():
    import smvp_toolkit_b200 as e

    if not os.path.exists(e.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return e


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _cuda(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


def _nan(n):
    import torch

    return torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")


def _band(m, offsets, rng):
    r = np.arange(m)
    rows = np.concatenate([r[(r + d >= 0) & (r + d < m)] for d in offsets])
    cols = np.concatenate([r[(r + d >= 0) & (r + d < m)] + d for d in offsets])
    return oracle.make_coo(rows, cols, rng.uniform(-1, 1, len(rows)))


def _matrices():
    """(name, m, n, coo, env): the shapes and plans the update has to keep"""
    rng = np.random.default_rng(5)
    coo = util.random_coo(rng, 400, 500, 3000)
    yield "random rectangular, empty rows and columns", 400, 500, coo[(coo["row"] % 7 != 0) & (coo["col"] % 5 != 0)], {}
    m, n, coo = util.load_sample("memplus")
    yield "memplus", m, n, coo, {}
    yield "stencil27 9x8x7", 9 * 8 * 7, 9 * 8 * 7, synth_ref.stencil27(9, 8, 7), {}
    yield "band (AUTO -> vector)", 3000, 3000, _band(3000, (-300, -2, -1, 0, 1, 2, 300), rng), {}
    coo = synth_ref.rmat(13, 12 << 13)
    yield "rmat 13 relabelled", 1 << 13, 1 << 13, coo, {"SMVP_CSR_RELABEL": "1", "SMVP_TJDS_RELABEL": "1"}


MATRICES = list(_matrices())


def _info(eng, A):
    """info fields an update must reproduce (all but input_order and device_bytes)"""
    csr = isinstance(A, eng.CsrMatrix)
    info = eng.engine._CsrInfo() if csr else eng.engine._TjdsInfo()
    fn = eng.lib().smvp_csr_info if csr else eng.lib().smvp_tjds_info
    assert fn(A._h, ctypes.byref(info)) == 0
    out = {f: getattr(info, f) for f, _ in info._fields_ if f not in ("input_order", "device_bytes")}
    out["launches_per_mult"] = list(out["launches_per_mult"])
    return out


def _device_bytes(eng, A):
    info = eng.engine._CsrInfo() if isinstance(A, eng.CsrMatrix) else eng.engine._TjdsInfo()
    fn = eng.lib().smvp_csr_info if isinstance(A, eng.CsrMatrix) else eng.lib().smvp_tjds_info
    assert fn(A._h, ctypes.byref(info)) == 0
    return info.device_bytes


def csr_passes(eng, A, dx, declare):
    """every pass of a CSR handle: each variant plain (declared x and explicit x), *_axpby, *_axpby_dot (w and ||y||^2),
    fan-out, and the host -n loop (exact and batched).  dx must stay alive: it is the declared x."""
    import torch

    rng = np.random.default_rng(1)
    m = A.rows
    if declare:
        A.set_x_device(dx)
    out = {}
    dw = _cuda(rng.uniform(-1, 1, m))
    for v in CSR_VARIANTS:
        dy = _nan(m)
        A.mult_device(None, dy, v)
        out["plain declared", v] = dy
        dy = _nan(m)
        A.mult_device(dx, dy, v)
        out["plain", v] = dy
        for a, b in PAIRS:
            y0 = rng.uniform(-2, 2, m)
            dy = _cuda(y0.copy())
            A.mult_device_axpby(a, None, b, dy, v)
            out["axpby", v, a, b] = dy
            for w in (None, dw):
                dy, dd = _cuda(y0.copy()), _nan(1)
                A.mult_device_axpby_dot(a, None, b, dy, w, dd, v)
                out["dot y", v, a, b, w is None] = dy
                out["dot", v, a, b, w is None] = dd
        fan = [_nan(m) for _ in range(2)]
        A.mult_device_fanout(dx, [f.data_ptr() for f in fan], v)
        for k, f in enumerate(fan):
            out["fan-out", v, k] = f
    torch.cuda.synchronize()
    out = {k: t.cpu().numpy() for k, t in out.items()}
    x = dx.cpu().numpy()
    for v in CSR_VARIANTS:
        for iters in (1, 5):
            out["host", v, iters] = A.mult(x, iters=iters, variant=v)[0]
    return out


def tjds_passes(eng, A, dx, dxt, declare):
    """every pass of a TJDS handle: each variant plain, *_axpby, *_axpby_dot; A^T x plain, *_axpby, *_axpby_dot; the host
    -n loops of both (the host loop declares its own copy of x, so it runs last)"""
    import torch

    rng = np.random.default_rng(2)
    m, n = A.rows, A.cols
    if declare:
        A.set_x_device(dx)
    out = {}
    dw = _cuda(rng.uniform(-1, 1, m))
    for v in TJDS_VARIANTS:
        dy = _nan(m)
        A.mult_device(dy, v)
        out["plain", v] = dy
        for a, b in PAIRS:
            y0 = rng.uniform(-2, 2, m)
            dy = _cuda(y0.copy())
            A.mult_device_axpby(a, b, dy, v)
            out["axpby", v, a, b] = dy
            for w in (None, dw):
                dy, dd = _cuda(y0.copy()), _nan(1)
                A.mult_device_axpby_dot(a, b, dy, w, dd, v)
                out["dot y", v, a, b, w is None] = dy
                out["dot", v, a, b, w is None] = dd
    dwt = _cuda(rng.uniform(-1, 1, n))
    dy = _nan(n)
    A.mult_transpose_device(dxt, dy)
    out["transposed"] = dy
    for a, b in PAIRS:
        y0 = rng.uniform(-2, 2, n)
        dy = _cuda(y0.copy())
        A.mult_transpose_device_axpby(a, dxt, b, dy)
        out["transposed axpby", a, b] = dy
        for w in (None, dwt):
            dy, dd = _cuda(y0.copy()), _nan(1)
            A.mult_transpose_device_axpby_dot(a, dxt, b, dy, w, dd)
            out["transposed dot y", a, b, w is None] = dy
            out["transposed dot", a, b, w is None] = dd
    torch.cuda.synchronize()
    out = {k: t.cpu().numpy() for k, t in out.items()}
    out["route"] = np.array(A.plan(), np.float64)
    x, xt = dx.cpu().numpy(), dxt.cpu().numpy()
    for v in TJDS_VARIANTS:
        for iters in (1, 5):
            out["host", v, iters] = A.mult(x, iters=iters, variant=v)[0]
    for iters in (1, 5):
        out["host transposed", iters] = A.mult_transpose(xt, iters=iters)[0]
    return out


def _atomic(key, route):
    """outputs of the atomic kernel (the atomic variant, and the deterministic ones routed to it): as reproducible as
    between two runs"""
    v = key[1] if isinstance(key, tuple) and len(key) > 1 and key[0] in ("plain", "axpby", "dot y", "dot", "host") else None
    return v == 0 or (v in (1, 2) and route == -1)


def compare(got, want, tjds=False):
    assert got.keys() == want.keys()
    route = want["route"][1] if tjds else 1
    for k in want:
        if tjds and _atomic(k, route):
            assert np.array_equal(np.isfinite(got[k]), np.isfinite(want[k])), k
            f = np.isfinite(want[k])
            assert util.rel_l2(got[k][f], want[k][f]) <= TOL, k
        else:
            assert np.array_equal(bits(got[k]), bits(want[k])), k


def _update_list(coo, rng, subset):
    """(updated COO, list): new values on every entry in shuffled order, or on a random third of them; explicit zeros
    among the new values"""
    idx = rng.permutation(len(coo))
    if subset:
        idx = idx[:len(coo) // 3]
    new = coo.copy()
    vals = rng.uniform(-4, 4, len(idx))
    vals[::11] = 0.0
    new["val"][idx] = vals
    return new, new[idx]


def _apply(A, lst, device):
    if device:
        A.update_values_device(_cuda(lst["row"].astype(np.int32)), _cuda(lst["col"].astype(np.int32)), _cuda(lst["val"].astype(np.float64)),
                               len(lst))
    else:
        A.update_values(lst)


# ---------------------------------------------------------------------------- CPU
def test_strerror_names_the_pattern_error(eng):
    assert eng.E_PATTERN == -6
    text = eng.lib().smvp_strerror(eng.E_PATTERN).decode()
    assert text != eng.lib().smvp_strerror(-99).decode() and "not stored" in text


# ---------------------------------------------------------------------------- 1. equivalence
EQUIV = [(fmt, case, subset, skew) for fmt in ("csr", "tjds") for case in range(len(MATRICES)) for subset in (False, True)
         for skew in ((None,) if fmt == "csr" else ("0", "1"))]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,case,subset,skew", EQUIV,
                         ids=["%s-%s-%s%s" % (f, MATRICES[c][0], "subset" if s else "all shuffled", "" if k is None else "-skew" + k)
                              for f, c, s, k in EQUIV])
def test_update_equals_a_fresh_build(eng, monkeypatch, fmt, case, subset, skew):
    """H0 runs every pass (every lazy plan and scratch exists), takes the update (host list for a full update, device
    list for a subset), runs the passes again on the x declared before the update; H1 is built from the updated COO and
    runs the same passes.  Exports, info and every output agree."""
    name, m, n, coo, env = MATRICES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    if skew is not None:
        monkeypatch.setenv("SMVP_TJDS_SKEW", skew)
    rng = np.random.default_rng(100 + case)
    dx, dxt = _cuda(rng.uniform(-1, 1, n)), _cuda(rng.uniform(-1, 1, m))
    new, lst = _update_list(coo, rng, subset)
    if fmt == "csr":
        H0 = eng.CsrMatrix.build(coo, m, n)
        csr_passes(eng, H0, dx, True)
        pointers = H0.device_arrays()
        _apply(H0, lst, subset)
        got = csr_passes(eng, H0, dx, False)
        H1 = eng.CsrMatrix.build(new, m, n)
        want = csr_passes(eng, H1, dx, True)
        assert H0.device_arrays() == pointers
        compare(got, want)
        if "RELABEL" in str(env):
            assert _info(eng, H0)["x_relabel"] == 1
    else:
        H0 = eng.TjdsMatrix.build(coo, m, n)
        tjds_passes(eng, H0, dx, dxt, True)
        _apply(H0, lst, subset)
        got = tjds_passes(eng, H0, dx, dxt, False)
        H1 = eng.TjdsMatrix.build(new, m, n)
        want = tjds_passes(eng, H1, dx, dxt, True)
        compare(got, want, tjds=True)
        assert _info(eng, H0)["skewed_walk"] == (1 if skew == "1" else -1)
        if "RELABEL" in str(env):
            assert _info(eng, H0)["y_relabel"] == 1
    for a, b in zip(H0.export(), H1.export()):
        assert np.array_equal(a.view(np.int64) if a.dtype == np.float64 else a, b.view(np.int64) if b.dtype == np.float64 else b)
    assert _info(eng, H0) == _info(eng, H1)
    H0.free()
    H1.free()


# ---------------------------------------------------------------------------- 2. width transitions
@pytest.mark.gpu
def test_width_transitions_of_the_row_pattern_plan(eng):
    """2 -> 8 -> 4 -> 2: value_bytes and device_bytes follow the values, the device array pointers never change, and
    every pass is bit-identical to a fresh build at each step."""
    rng = np.random.default_rng(7)
    m = 9 * 8 * 7
    coo = synth_ref.stencil27(9, 8, 7)  # {26, -1}: fp16
    dx = _cuda(rng.uniform(-1, 1, m))
    A = eng.CsrMatrix.build(coo, m, m)
    csr_passes(eng, A, dx, True)
    assert A.row_patterns == 27 and A.value_bytes == 2
    pointers = A.device_arrays()
    narrow = lambda w: w * len(coo) if w < 8 else 0  # noqa: E731
    width = 2
    for want_w, vals in ((8, rng.uniform(-1, 1, len(coo))), (4, rng.uniform(-1, 1, len(coo)).astype(np.float32).astype(np.float64)),
                         (2, rng.integers(-9, 10, len(coo)).astype(np.float64))):
        new = coo.copy()
        new["val"] = vals
        before = _device_bytes(eng, A)
        A.update_values(new[rng.permutation(len(new))])
        assert A.value_bytes == want_w
        assert _device_bytes(eng, A) - before == narrow(want_w) - narrow(width)
        assert A.device_arrays() == pointers
        got = csr_passes(eng, A, dx, False)
        B = eng.CsrMatrix.build(new, m, m)
        compare(got, csr_passes(eng, B, dx, True))
        assert _info(eng, A) == _info(eng, B)
        B.free()
        width = want_w
    A.free()


# ---------------------------------------------------------------------------- 3. partial update: A - sigma I
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "tjds"])
def test_shift_of_the_diagonal(eng, fmt):
    """Updating only the stored diagonal entries (A - sigma I) equals a fresh build of the shifted matrix."""
    rng = np.random.default_rng(8)
    for name, m, n, coo, _ in (MATRICES[1], MATRICES[2]):
        diag = np.flatnonzero(coo["row"] == coo["col"])
        assert len(diag) > 0, name
        new = coo.copy()
        new["val"][diag] -= 0.75
        dx, dxt = _cuda(rng.uniform(-1, 1, n)), _cuda(rng.uniform(-1, 1, m))
        if fmt == "csr":
            A, B = eng.CsrMatrix.build(coo, m, n), eng.CsrMatrix.build(new, m, n)
            csr_passes(eng, A, dx, True)
            A.update_values(new[diag])
            compare(csr_passes(eng, A, dx, False), csr_passes(eng, B, dx, True))
        else:
            A, B = eng.TjdsMatrix.build(coo, m, n), eng.TjdsMatrix.build(new, m, n)
            tjds_passes(eng, A, dx, dxt, True)
            A.update_values(new[diag])
            compare(tjds_passes(eng, A, dx, dxt, False), tjds_passes(eng, B, dx, dxt, True), tjds=True)
        for a, b in zip(A.export(), B.export()):
            assert np.array_equal(a, b) if a.dtype != np.float64 else np.array_equal(bits(a), bits(b))
        A.free()
        B.free()


# ---------------------------------------------------------------------------- 4. TJDS routing
@pytest.mark.gpu
def test_tjds_route_follows_the_values(eng):
    """With x declared once, before the updates: an Inf sends the deterministic variant to the atomic kernel, a row of
    zeros only turns the short split loop off, finite nonzero values restore both -- in each state as on a fresh build
    with the same x."""
    rng = np.random.default_rng(9)
    m, n = 500, 300
    coo = util.random_coo(rng, m, n, 6000)
    dx = _cuda(rng.uniform(-1, 1, n))
    A = eng.TjdsMatrix.build(coo, m, n)
    A.set_x_device(dx)
    dy = _nan(m)
    assert det_kernel_fast_flags(lambda: A.mult_device(dy, 1)) == [True] and A.plan()[1] == 1  # the state an update revises
    row = int(coo["row"][0])
    in_row = np.flatnonzero(coo["row"] == row)
    inf = coo.copy()
    inf["val"][5] = np.inf
    zero_row = coo.copy()
    zero_row["val"][in_row] = 0.0
    states = [("inf", inf, -1, []), ("zero row", zero_row, 1, [False]), ("finite", coo, 1, [True])]
    for name, new, route, fast in states:
        A.update_values(new[rng.permutation(len(new))])
        assert A.plan()[1] == 0, name  # decided again at the next pass
        B = eng.TjdsMatrix.build(new, m, n)
        B.set_x_device(dx)
        ys = []
        for H in (A, B):
            dy = _nan(m)
            flags = det_kernel_fast_flags(lambda: H.mult_device(dy, 1))
            ys.append(dy.cpu().numpy())
            assert H.plan()[1] == route and flags == fast, (name, H is A, H.plan(), flags)
        if route == 1:
            assert np.array_equal(bits(ys[0]), bits(ys[1])), name
        else:
            assert np.array_equal(np.isfinite(ys[0]), np.isfinite(ys[1])) and (~np.isfinite(ys[0])).any(), name
            f = np.isfinite(ys[0])
            assert util.rel_l2(ys[0][f], ys[1][f]) <= TOL, name
        B.free()
    A.free()


# ---------------------------------------------------------------------------- 5. errors
def _snapshot(eng, A, dx):
    import torch

    dy = _nan(A.rows)
    if isinstance(A, eng.CsrMatrix):
        A.mult_device(None, dy, 2)
    else:
        A.mult_device(dy, 1)
    torch.cuda.synchronize()
    return [a.view(np.int64) if a.dtype == np.float64 else a for a in A.export()] + [bits(dy.cpu().numpy())], _info(eng, A)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "tjds"])
def test_rejected_lists_leave_the_handle_untouched(eng, fmt):
    """The offending entry is the last of a long list: E_RANGE, E_PATTERN and the E_ARG cases change neither the arrays
    nor y nor info; n = 0 is a no-op; a handle without entries rejects any pair with E_PATTERN."""
    rng = np.random.default_rng(10)
    m = 9 * 8 * 7
    coo = synth_ref.stencil27(9, 8, 7)
    coo["val"] = rng.uniform(-1, 1, len(coo))
    dx = _cuda(rng.uniform(-1, 1, m))
    cls = eng.CsrMatrix if fmt == "csr" else eng.TjdsMatrix
    L = eng.lib()
    upd, upd_dev = ((L.smvp_csr_update_values, L.smvp_csr_update_values_device) if fmt == "csr" else
                    (L.smvp_tjds_update_values, L.smvp_tjds_update_values_device))
    A = cls.build(coo, m, m)
    A.set_x_device(dx)
    before = _snapshot(eng, A, dx)
    good = coo[rng.permutation(len(coo))].copy()
    good["val"] = rng.uniform(-1, 1, len(good))
    stored = set(zip(coo["row"].tolist(), coo["col"].tolist()))
    assert (0, m - 1) not in stored
    for bad, code in (((m, 0), eng.E_RANGE), ((0, m), eng.E_RANGE), ((-1, 3), eng.E_RANGE), ((0, m - 1), eng.E_PATTERN)):
        lst = np.concatenate([good, oracle.make_coo(np.array([bad[0]]), np.array([bad[1]]), np.array([7.0]))])
        with pytest.raises(eng.SmvpError) as ei:
            A.update_values(lst)
        assert ei.value.code == code, bad
        with pytest.raises(eng.SmvpError) as ei:
            _apply(A, lst, True)
        assert ei.value.code == code, bad
        after = _snapshot(eng, A, dx)
        assert all(np.array_equal(a, b) for a, b in zip(after[0], before[0])) and after[1] == before[1], bad
    p = eng.engine._ptr
    dr, dc, dv = _cuda(good["row"].astype(np.int32)), _cuda(good["col"].astype(np.int32)), _cuda(good["val"].astype(np.float64))
    assert upd(None, p(good), len(good)) == eng.E_ARG
    assert upd(A._h, p(good), -1) == eng.E_ARG
    assert upd(A._h, None, 3) == eng.E_ARG
    assert upd_dev(None, p(dr), p(dc), p(dv), len(good), None) == eng.E_ARG
    assert upd_dev(A._h, p(dr), p(dc), p(dv), -1, None) == eng.E_ARG
    for k in range(3):
        args = [p(dr), p(dc), p(dv)]
        args[k] = None
        assert upd_dev(A._h, *args, len(good), None) == eng.E_ARG, k
    assert upd(A._h, None, 0) == eng.OK and upd_dev(A._h, None, None, None, 0, None) == eng.OK
    A.update_values(good[:0])
    after = _snapshot(eng, A, dx)
    assert all(np.array_equal(a, b) for a, b in zip(after[0], before[0])) and after[1] == before[1]
    A.free()

    E = cls.build(oracle.make_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0)), 30, 40)
    with pytest.raises(eng.SmvpError) as ei:
        E.update_values(oracle.make_coo(np.array([1]), np.array([2]), np.array([3.0])))
    assert ei.value.code == eng.E_PATTERN
    assert upd(E._h, None, 0) == eng.OK
    E.free()


# ---------------------------------------------------------------------------- 6. transpose
@pytest.mark.gpu
@pytest.mark.parametrize("case", [0, 3], ids=[MATRICES[0][0], MATRICES[3][0]])
def test_transposed_handle_takes_the_swapped_list(eng, case):
    """smvp_csr_transpose(A) updated with the list with rows and columns swapped == smvp_csr_transpose of the updated A:
    the same arrays and the same A^T x bits from every pass."""
    name, m, n, coo, _ = MATRICES[case]
    rng = np.random.default_rng(11)
    dxt = _cuda(rng.uniform(-1, 1, m))
    A = eng.CsrMatrix.build(coo, m, n)
    T = A.transpose()
    csr_passes(eng, T, dxt, True)
    new, lst = _update_list(coo, rng, True)
    A.update_values(lst)
    T.update_values(oracle.make_coo(lst["col"], lst["row"], lst["val"]))
    T2 = A.transpose()
    compare(csr_passes(eng, T, dxt, False), csr_passes(eng, T2, dxt, True))
    for a, b in zip(T.export(), T2.export()):
        assert np.array_equal(a, b) if a.dtype != np.float64 else np.array_equal(bits(a), bits(b))
    for H in (A, T, T2):
        H.free()


# ---------------------------------------------------------------------------- 7. no rebuild
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "tjds"])
def test_update_launches_do_not_grow_with_the_matrix(eng, fmt):
    """The launches of an update are the same for two stencils whose nnz differ by more than 100x, and fewer than a
    build's."""
    import torch

    counts = []
    for nx in (8, 38):
        m = nx ** 3
        r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH)
        assert nx == 8 or r.n > 100 * counts[0][2]
        cls = eng.CsrMatrix if fmt == "csr" else eng.TjdsMatrix
        b0 = eng.launch_count()
        A = cls.build_device(r, c, v, m, m, r.n)
        built = eng.launch_count() - b0
        dx = _cuda(np.ones(m))
        dy = _nan(m)
        if fmt == "csr":
            A.mult_device(dx, dy, 2)
            assert A.row_patterns == 27
        else:
            A.set_x_device(dx)
            A.mult_device(dy, 1)
            assert A.plan()[1] == 1
        torch.cuda.synchronize()
        u0 = eng.launch_count()
        A.update_values_device(r, c, v, r.n)
        counts.append((eng.launch_count() - u0, built, r.n))
        A.free()
        for a in (r, c, v):
            a.free()
    assert counts[0][0] == counts[1][0] and counts[0][0] < min(counts[0][1], counts[1][1]), counts
