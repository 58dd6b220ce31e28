"""Deterministic TJDS (SMVP_TJDS_DETERMINISTIC and SMVP_TJDS_DETERMINISTIC_FAST) bit for bit against an exact model of
the integer accumulation, the contract stated in include/smvp_cuda.h:

    e(v)   the frexp exponent of v (ilogb(v) + 1): |v| < 2^e(v)
    ea_r   max e(a_rj) over the nonzero entries of row r
    cb_r   ceil(log2 count_r), counting every stored entry of row r, explicit zeros included
    ex     max e(x_c) over the nonzero x_c of the columns that hold entries
    T_r  = ea_r + cb_r + ex
    p    = fl(a * x)
    y_r  = RN( sum_j trunc0(p_j * 2^(F - T_r)) * 2^(T_r - F) ),   F = 94 (DETERMINISTIC) or 62 (DETERMINISTIC_FAST)

trunc0 truncates toward zero, the sum is exact (Python integers) and RN is ONE round-to-nearest-even to fp64, subnormal
results included (int / int true division rounds correctly).  Rows without a nonzero product are +0.0.  The kernels
split trunc0(p * 2^(94 - T_r)) into a high word trunc0(p * 2^(62 - T_r)) and a 32-bit low word, both signed like p,
and add each kind in a 64-bit integer accumulator; DETERMINISTIC rounds (sum hi) * 2^32 + (sum lo), FAST the high words
alone.  The model keeps the same two sums, so that it can also restate the conversion the library used before it
rounded once (fl(fl(hi) * 2^32 + lo)), which the double-rounding case must tell apart.

Where every nonzero product is a multiple of 2^(T_r - 94) (for instance |p| >= 2^(T_r - 42)) the model is the correctly
rounded row sum, math.fsum; otherwise it is within 1/2 ulp(y_r) + count_r * 2^(T_r - 94) of the exact sum."""
import math
import re
from fractions import Fraction

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle

DET, FAST = 1, 2  # SMVP_TJDS_DETERMINISTIC, SMVP_TJDS_DETERMINISTIC_FAST
FRAC = 94  # value = V * 2^(T - FRAC) for the two-word sum V = hi * 2^W + lo
W = 32  # bits of the low word


# ---------------------------------------------------------------------------- the model, in Python integers
def fexp(v):
    """e(v): the frexp exponent, |v| < 2^e(v), for v != 0 (subnormals included)"""
    return math.frexp(v)[1]


def ceil_log2(c):
    return (c - 1).bit_length() if c > 1 else 0


def trunc_scaled(p, s):
    """trunc0(p * 2^s) as a Python integer"""
    n, d = abs(p).as_integer_ratio()  # d is a power of two
    t = (n << s) // d if s >= 0 else n // (d << -s)
    return -t if p < 0 else t


def split(p, T):
    """(hi, lo) words of trunc0(p * 2^(94 - T)): hi = trunc0(p * 2^(62 - T)), lo the remaining 32 bits, both signed like p"""
    v = trunc_scaled(p, FRAC - T)
    h = abs(v) >> W
    h = -h if v < 0 else h
    return h, v - (h << W)


def rn(v, e):
    """v * 2^e rounded once to nearest even fp64"""
    return float(v << e) if e >= 0 else v / (1 << -e)


def row_bounds(coo, m, x):
    """T_r for every row (None: the row holds no nonzero value, or x is zero on every column that holds an entry)"""
    cols = np.unique(coo["col"])
    xe = [fexp(v) for v in x[cols].tolist() if v != 0.0]
    if not xe:
        return [None] * m
    ex = max(xe)
    ea, cnt = [None] * m, [0] * m
    for r, a in zip(coo["row"].tolist(), coo["val"].tolist()):
        cnt[r] += 1
        if a != 0.0:
            ea[r] = fexp(a) if ea[r] is None else max(ea[r], fexp(a))
    return [None if ea[r] is None else ea[r] + ceil_log2(cnt[r]) + ex for r in range(m)]


def model_words(coo, m, x, walked=None):
    """(T, H, L): row bounds and, per row, the exact integer sums of the high and low words.  `walked` (a COO of a subset
    of the entries, e.g. the diagonals a diag_limit pass visits) is summed instead of `coo`; the bounds come from coo."""
    T = row_bounds(coo, m, x)
    s = coo if walked is None else walked
    prods = s["val"] * x[s["col"]]  # fl(a * x): numpy multiplies in IEEE fp64, round to nearest, no FMA
    H, L = [0] * m, [0] * m
    for r, p in zip(s["row"].tolist(), prods.tolist()):
        if p != 0.0:
            h, lo = split(p, T[r])
            H[r] += h
            L[r] += lo
    return T, H, L


def model(coo, m, x, variant, walked=None):
    """y of the deterministic variant: one rounding of the exact sum of the truncated products"""
    T, H, L = model_words(coo, m, x, walked)
    y = np.zeros(m)
    for r in range(m):
        if T[r] is not None:
            y[r] = rn((H[r] << W) + L[r], T[r] - FRAC) if variant == DET else rn(H[r], T[r] - (FRAC - W))
    return y


def parent_conversion(coo, m, x):
    """DETERMINISTIC as converted before the single rounding: fl(fl(hi) * 2^32 + lo) * 2^(T - 94)"""
    T, H, L = model_words(coo, m, x)
    y = np.zeros(m)
    for r in range(m):
        if H[r] or L[r]:
            y[r] = math.ldexp(float(H[r]) * 2.0 ** W + float(L[r]), T[r] - FRAC)
    return y


def fsum_rows(coo, m, x):
    y = np.zeros(m)
    prods = coo["val"] * x[coo["col"]]
    order = np.argsort(coo["row"], kind="stable")
    rows, prods = coo["row"][order], prods[order]
    bounds = np.searchsorted(rows, np.arange(m + 1))
    for r in range(m):
        y[r] = math.fsum(prods[bounds[r]:bounds[r + 1]].tolist())
    return y


# ---------------------------------------------------------------------------- the model on int64 words, in numpy
def split_np(p, T):
    """split() for arrays: (hi, lo) int64 words of trunc0(p * 2^(94 - T)) from the fp64 fields of p, as fixed_split in
    tjds_mult.cu computes them (V = m * 2^s, |V| < 2^94, never formed as one integer)"""
    bits = np.ascontiguousarray(p, np.float64).view(np.int64)
    be = (bits >> 52) & 0x7FF
    mant = ((bits & ((1 << 52) - 1)) | np.where(be > 0, 1 << 52, 0)).astype(np.uint64)
    e = np.where(be > 0, be - 1075, -1074)
    s = e - (np.asarray(T, np.int64) - FRAC)
    mask = np.uint64((1 << W) - 1)

    def sh(v, k, left):  # v << k or v >> k for k in [0, 63]
        k = np.clip(k, 0, 63).astype(np.uint64)
        return np.left_shift(v, k) if left else np.right_shift(v, k)

    t = sh(mant, -s, False)  # s < 0: the bits of V
    hm = np.where(s >= W, sh(mant, s - W, True), np.where(s >= 0, sh(mant, W - s, False), t >> np.uint64(W)))
    lm = np.where(s >= W, np.uint64(0), np.where(s >= 0, sh(mant, s, True) & mask, t & mask))
    hm = np.where(s <= -64, np.uint64(0), hm).astype(np.int64)
    lm = np.where(s <= -64, np.uint64(0), lm).astype(np.int64)
    neg = bits < 0
    return np.where(neg, -hm, hm), np.where(neg, -lm, lm)


def model_np(coo, m, x, variants=(DET, FAST)):
    """{variant: y} for a large COO: the split on int64 words, the exact per-row sums with np.add.at (int64 cannot
    overflow under the row bound: |sum hi| <= 2^62, |sum lo| < count * 2^32), one rounding per row in Python integers"""
    rows, cols, vals = coo["row"].astype(np.int64), coo["col"].astype(np.int64), coo["val"]
    used = np.zeros(len(x), bool)
    used[cols] = True
    xn = x[used & (x != 0)]
    out = {v: np.zeros(m) for v in variants}
    if len(xn) == 0:
        return out
    ex = int(np.frexp(xn)[1].max())
    nz = vals != 0
    ea = np.full(m, np.iinfo(np.int64).min // 2)
    np.maximum.at(ea, rows[nz], np.frexp(vals[nz])[1].astype(np.int64))
    cnt = np.bincount(rows, minlength=m)
    cb = np.array([ceil_log2(int(c)) for c in cnt], np.int64)
    T = ea + cb + ex
    p = vals * x[cols]
    hi, lo = split_np(p, T[rows])
    H, L = np.zeros(m, np.int64), np.zeros(m, np.int64)
    np.add.at(H, rows, hi)
    np.add.at(L, rows, lo)
    for r in np.flatnonzero((H != 0) | (L != 0)).tolist():
        if DET in out:
            out[DET][r] = rn((int(H[r]) << W) + int(L[r]), int(T[r]) - FRAC)
        if FAST in out:
            out[FAST][r] = rn(int(H[r]), int(T[r]) - (FRAC - W))
    return out


# ---------------------------------------------------------------------------- data sets
def existing_data():
    """rows with products over 16 decades: the data of the suite's first exactness check"""
    rng = np.random.default_rng(5)
    m, n, nnz = 400, 400, 20000
    coo = util.random_coo(rng, m, n, nnz)
    coo["val"] *= 10.0 ** rng.integers(-8, 8, nnz)
    x = rng.uniform(-1, 1, n) * 10.0 ** rng.integers(-3, 3, n)
    return coo, m, n, x


def double_rounding_rows(count=100, length=3, n=16):
    """`count` rows of `length` entries, x = ones, on which fl(fl(hi) * 2^32 + lo) differs from RN(hi * 2^32 + lo): the
    first such rows of a fixed random stream (values of one sign or mixed, magnitudes over 30 binades)"""
    rng = np.random.default_rng(2024)
    x = np.ones(n)
    found = []
    while len(found) < count:
        cols = rng.choice(n, size=length, replace=False)
        vals = rng.uniform(0.5, 1.0, length) * 2.0 ** rng.integers(-30, 1, length) * rng.choice([-1.0, 1.0, 1.0], length)
        coo = oracle.make_coo(np.zeros(length, np.int64), cols, vals)
        if parent_conversion(coo, 1, x)[0] != model(coo, 1, x, DET)[0]:
            found.append((cols, vals))
    rows = np.repeat(np.arange(count), length)
    coo = oracle.make_coo(rows, np.concatenate([c for c, _ in found]), np.concatenate([v for _, v in found]))
    return coo, count, n, x


def random_rows(rng, nrows, spread):
    """rows of 1..64 entries whose value exponents span `spread` binades and x in [1/2, 1)"""
    rows, cols, vals = [], [], []
    for r in range(nrows):
        k = int(rng.integers(1, 65))
        rows += [r] * k
        cols += rng.choice(64, size=k, replace=False).tolist()
        vals += (rng.uniform(0.5, 1.0, k) * 2.0 ** rng.integers(-spread, 1, k) * rng.choice([-1.0, 1.0], k)).tolist()
    return oracle.make_coo(np.array(rows), np.array(cols), np.array(vals)), nrows, 64, rng.uniform(0.5, 1.0, 64)


# ---------------------------------------------------------------------------- CPU: the model itself
def test_model_is_fsum_where_every_product_is_on_the_grid():
    """|p| >= 2^(T_r - 42) makes p a multiple of 2^(T_r - 94): nothing is truncated, the model is the correctly rounded sum"""
    rng = np.random.default_rng(11)
    checked = 0
    for spread in (8, 30, 60):
        coo, m, n, x = random_rows(rng, 1500, spread)
        T = row_bounds(coo, m, x)
        p = coo["val"] * x[coo["col"]]
        on_grid = np.ones(m, bool)
        for r, v in zip(coo["row"].tolist(), p.tolist()):
            if v != 0.0 and abs(v) < 2.0 ** (T[r] - 42):
                on_grid[r] = False
        want = fsum_rows(coo, m, x)
        got = model(coo, m, x, DET)
        assert np.array_equal(util_bits(got[on_grid]), util_bits(want[on_grid]))
        checked += int(on_grid.sum())
    assert checked >= 3000


def test_model_drops_exactly_the_truncated_bits():
    """{1, -1, 2^-100} with x = ones: T = 1 + 2 + 1, the truncation at 2^-90 drops 2^-100, the sum of what is kept is 0"""
    coo = oracle.make_coo([0, 0, 0], [0, 1, 2], [1.0, -1.0, 2.0 ** -100])
    x = np.ones(3)
    assert row_bounds(coo, 1, x) == [4]
    y = model(coo, 1, x, DET)[0]
    assert util_bits(y) == 0 and math.fsum([1.0, -1.0, 2.0 ** -100]) == 2.0 ** -100
    # in general: exact sum - kept sum = the bits below 2^(T - 94), per product
    rng = np.random.default_rng(3)
    coo, m, n, x = random_rows(rng, 300, 200)
    T, H, L = model_words(coo, m, x)
    dropped, exact = [Fraction(0)] * m, [Fraction(0)] * m
    for r, p in zip(coo["row"].tolist(), (coo["val"] * x[coo["col"]]).tolist()):
        h, lo = split(p, T[r])
        exact[r] += Fraction(p)
        dropped[r] += Fraction(p) - Fraction((h << W) + lo) * Fraction(2) ** (T[r] - FRAC)
    for r in range(m):
        kept = Fraction((H[r] << W) + L[r]) * Fraction(2) ** (T[r] - FRAC)
        assert exact[r] - kept == dropped[r]
        assert abs(dropped[r]) < Fraction(64) * Fraction(2) ** (T[r] - FRAC)


def test_numpy_split_is_the_integer_split():
    rng = np.random.default_rng(8)
    k = 20000
    p = rng.uniform(-1, 1, k) * 2.0 ** rng.integers(-1074, 1000, k)
    p[:50] = np.array([5e-324, -5e-324, 2.0 ** -1022, -(2.0 ** -1023) * 1.5, 0.0, -0.0] * 8 + [1.0, -1.0])
    # bounds from "p is the whole row" up to 200 binades above p, and the general split's range below -929
    T = np.array([fexp(v) if v != 0.0 else 0 for v in p.tolist()]) + rng.integers(0, 200, k)
    hi, lo = split_np(p, T)
    for i in range(k):
        assert (int(hi[i]), int(lo[i])) == split(float(p[i]), int(T[i])), (p[i], T[i])
    coo, m, n, x = band_data()
    want = model_np(coo, m, x)
    for v in (DET, FAST):
        assert np.array_equal(util_bits(want[v]), util_bits(model(coo, m, x, v)))


def test_existing_data_model_is_fsum_and_parent_conversion_is_not():
    """On the suite's first exactness data every product is on its row's grid, so the model is math.fsum; the conversion
    that rounded hi on its own was 1 ulp off on some of these rows"""
    coo, m, n, x = existing_data()
    want = fsum_rows(coo, m, x)
    assert np.array_equal(util_bits(model(coo, m, x, DET)), util_bits(want))
    old = parent_conversion(coo, m, x)
    moved = np.flatnonzero(util_bits(old) != util_bits(want))
    assert len(moved) > 0
    assert np.all(np.abs(old[moved] - want[moved]) == np.spacing(np.abs(want[moved])))


def test_double_rounding_rows_are_found():
    coo, m, n, x = double_rounding_rows()
    assert np.all(util_bits(parent_conversion(coo, m, x)) != util_bits(model(coo, m, x, DET)))
    assert np.array_equal(util_bits(model(coo, m, x, DET)), util_bits(fsum_rows(coo, m, x)))


def util_bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


# ---------------------------------------------------------------------------- GPU: the library against the model
@pytest.fixture(scope="module")
def eng():
    import smvp_toolkit_b200 as e

    assert e.device_count() >= 1
    return e


def _cuda(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a, np.float64), device="cuda")


def same_bits(got, want, what=""):
    got, want = util_bits(got), util_bits(want)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, "%s: %d rows differ, first %s" % (what, len(bad), bad[:8].tolist())


def check_host(eng, coo, m, n, x, variants=(DET, FAST), walked=None, diag_limit=0):
    """smvp_tjds_mult (host vectors) equals the model bit for bit and takes the integer path (det_route 1)"""
    A = eng.TjdsMatrix.build(coo, m, n)
    for v in variants:
        y, _ = A.mult(x, 1, v, diag_limit)
        assert A.plan()[1] == 1
        same_bits(y, model(coo, m, x, v, walked), "variant %d" % v)
    A.free()


@pytest.mark.gpu
def test_existing_data_is_bit_exact(eng):
    """rows whose products span 16 decades: every product is on its row's grid, so y is math.fsum bit for bit"""
    coo, m, n, x = existing_data()
    check_host(eng, coo, m, n, x)
    A = eng.TjdsMatrix.build(coo, m, n)
    y, _ = A.mult(x, 1, DET)
    same_bits(y, fsum_rows(coo, m, x), "fsum")
    A.free()


@pytest.mark.gpu
def test_double_rounding_rows_round_once(eng):
    """rows on which converting hi on its own and then adding lo rounds twice (1 ulp off the correctly rounded sum)"""
    coo, m, n, x = double_rounding_rows()
    check_host(eng, coo, m, n, x)


@pytest.mark.gpu
def test_truncation_follows_the_contract(eng):
    rng = np.random.default_rng(17)
    # the cancellation row: 1 - 1 + 2^-100 truncates to +0.0 (T = 4, the grid is 2^-90)
    coo = oracle.make_coo([0, 0, 0], [0, 1, 2], [1.0, -1.0, 2.0 ** -100])
    check_host(eng, coo, 1, 3, np.ones(3))
    # row 0: 27 O(1) products; row 1 reads the column of x that holds 1e12 / 1e20, which sets ex for every row
    for big in (1e12, 1e20):
        vals = np.concatenate([rng.uniform(-1, 1, 27), [0.75]])
        coo = oracle.make_coo([0] * 27 + [1], list(range(1, 28)) + [0], vals)
        x = np.concatenate([[big], rng.uniform(-1, 1, 27)])
        y = model(coo, 2, x, DET)
        assert y[0] != fsum_rows(coo, 2, x)[0]  # the truncation shows
        check_host(eng, coo, 2, 28, x)
    # a row spanning 2^-1000 .. 1
    k = np.arange(0, 1001, 9)
    vals = rng.uniform(0.5, 1.0, len(k)) * 2.0 ** -k.astype(np.float64) * rng.choice([-1.0, 1.0], len(k))
    coo = oracle.make_coo(np.zeros(len(k), np.int64), np.arange(len(k)), vals)
    check_host(eng, coo, 1, len(k), rng.uniform(0.5, 1.0, len(k)))


@pytest.mark.gpu
def test_x_entries_the_matrix_never_reads_do_not_change_y(eng):
    """x[c] of a column that holds no entry (1e30, Inf) gives the same bits as x[c] = 0, on the integer path"""
    rng = np.random.default_rng(23)
    m, n = 300, 400
    coo = util.random_coo(rng, m, n, 6000)
    coo = coo[coo["col"] % 10 != 3]  # columns 3, 13, ... hold no entry
    coo["val"] *= 10.0 ** rng.integers(-6, 6, len(coo))
    x0 = rng.uniform(-1, 1, n)
    x0[3::10] = 0.0
    A = eng.TjdsMatrix.build(coo, m, n)
    for v in (DET, FAST):
        y0, _ = A.mult(x0, 1, v)
        same_bits(y0, model(coo, m, x0, v), "x0")
        for big in (1e30, np.inf):
            x = x0.copy()
            x[13] = big
            y, _ = A.mult(x, 1, v)
            assert A.plan()[1] == 1, (v, big)
            same_bits(y, y0, "x[13] = %r" % big)
    A.free()


@pytest.mark.gpu
def test_general_split(eng):
    """Row bounds where 2^(94 - T) is not a normal double (T < -929): the integer split fixed_split, not the fp64 one"""
    rng = np.random.default_rng(29)
    n = 40
    rows, cols, vals = [], [], []

    def row(v):
        r = len(set(rows))
        k = len(v)
        rows.extend([r] * k)
        cols.extend(rng.choice(n, size=k, replace=False).tolist())
        vals.extend(v)

    for _ in range(20):  # values near 2^-990, x ~ 1: T < -929
        row((rng.uniform(-1, 1, 9) * 2.0 ** rng.integers(-1000, -985, 9)).tolist())
    for _ in range(20):  # subnormal values
        row((rng.integers(-2 ** 40, 2 ** 40, 7) * 5e-324).tolist())
    row([2.0 ** -1074, -(2.0 ** -1074), 3 * 2.0 ** -1074])
    coo = oracle.make_coo(np.array(rows), np.array(cols), np.array(vals))
    m = len(set(rows))
    x = rng.uniform(0.5, 2.0, n) * rng.choice([-1.0, 1.0], n)
    check_host(eng, coo, m, n, x)
    # products that underflow to a subnormal or to zero: values ~2^-540, x ~2^-520 .. 2^-560
    coo2 = util.random_coo(rng, 50, n, 600)
    coo2["val"] *= 2.0 ** -540
    x2 = rng.uniform(-1, 1, n) * 2.0 ** rng.integers(-560, -520, n)
    p = coo2["val"] * x2[coo2["col"]]
    assert (p == 0).any() and ((p != 0) & (np.abs(p) < 2.0 ** -1022)).any()
    check_host(eng, coo2, 50, n, x2)


def det_kernel_fast_flags(fn):
    """The FAST template argument of every tjds_det_kernel that fn launches, from the kernel names torch.profiler records"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    flags = []
    for ev in prof.events():
        k = (re.search(r"tjds_det_kernel<\s*\d+,\s*(?:true|false),\s*(true|false),", ev.name) or
             re.search(r"tjds_det_kernelILi\d+ELb[01]ELb([01])E", ev.name))
        if k:
            flags.append(k.group(1) in ("true", "1"))
    return flags


@pytest.mark.gpu
def test_zeros_empty_rows_and_the_general_kernel(eng, monkeypatch):
    """Explicit zero values (counted in cb_r), x with zeros, an all-zero x (every row +0.0) and empty rows, on the short
    loop (tjds_det_kernel<.., FAST = true>) and on the general loop, which SMVP_TJDS_DET_GENERAL forces and a row
    holding entries but no nonzero value selects by itself: both give the model's bits"""
    import torch

    rng = np.random.default_rng(31)
    m, n = 500, 300
    coo = util.random_coo(rng, m, n, 8000)
    coo = coo[coo["row"] % 7 != 2]  # empty rows
    coo["val"][rng.random(len(coo)) < 0.1] = 0.0
    coo["val"] *= 10.0 ** rng.integers(-5, 5, len(coo))
    assert np.array_equal(np.unique(coo["row"]), np.unique(coo["row"][coo["val"] != 0]))  # no row of zeros only
    x = rng.uniform(-1, 1, n)
    x[rng.random(n) < 0.2] = 0.0
    ys = {}
    for general in (False, True):
        if general:
            monkeypatch.setenv("SMVP_TJDS_DET_GENERAL", "1")
        else:
            monkeypatch.delenv("SMVP_TJDS_DET_GENERAL", raising=False)
        A = eng.TjdsMatrix.build(coo, m, n)
        A.set_x_device(_cuda(x))
        for v in (DET, FAST):
            want = model(coo, m, x, v)
            dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
            flags = det_kernel_fast_flags(lambda: A.mult_device(dy, v))
            assert flags and all(f == (not general) for f in flags), (v, general, flags)
            same_bits(dy.cpu().numpy(), want, "device, variant %d general %s" % (v, general))
            ys[(v, general)] = dy.cpu().numpy()
            y, _ = A.mult(x, 1, v)
            same_bits(y, want, "host, variant %d general %s" % (v, general))
            yz, _ = A.mult(np.zeros(n), 1, v)
            assert A.plan()[1] == 1 and np.all(util_bits(yz) == 0)  # +0.0
            y, _ = A.mult(x, 1, v)  # and back
            same_bits(y, want, "after x = 0, variant %d general %s" % (v, general))
        A.free()
    monkeypatch.delenv("SMVP_TJDS_DET_GENERAL")
    for v in (DET, FAST):
        same_bits(ys[(v, True)], ys[(v, False)], "general vs short loop, variant %d" % v)
    # a row holding entries but no nonzero value: the general loop without the variable
    z = coo.copy()
    z["val"][z["row"] == 5] = 0.0
    assert (z["row"] == 5).any()
    A = eng.TjdsMatrix.build(z, m, n)
    A.set_x_device(_cuda(x))
    for v in (DET, FAST):
        dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
        flags = det_kernel_fast_flags(lambda: A.mult_device(dy, v))
        assert flags and not any(flags), (v, flags)
        same_bits(dy.cpu().numpy(), model(z, m, x, v), "row of zeros, variant %d" % v)
    A.free()


@pytest.mark.gpu
def test_route_boundary(eng):
    """ex + max row bound = 1000 stays on the integer path with the model's bits; 1001 goes to the atomic kernel"""
    vals = [1.5 * 2.0 ** 497, -1.25 * 2.0 ** 496, 1.75 * 2.0 ** 497, 2.0 ** 400]  # ea = 498, cb = 2
    coo = oracle.make_coo([0, 0, 0, 0, 1], [0, 1, 2, 3, 4], vals + [3.0])
    for ex, route in ((500, 1), (501, -1)):
        x = np.array([0.625, -0.875, 0.75, 0.5625, -0.9375]) * 2.0 ** ex  # max e(x) = ex
        A = eng.TjdsMatrix.build(coo, 2, 5)
        for v in (DET, FAST):
            y, _ = A.mult(x, 1, v)
            assert A.plan()[1] == route, (ex, v)
            if route == 1:
                same_bits(y, model(coo, 2, x, v), "ex %d" % ex)
        A.free()


def band_data(seed=37, m=3000):
    """a banded matrix (runs for the skewed walk) with products over 16 decades and a few rows that round twice"""
    rng = np.random.default_rng(seed)
    r = np.arange(m)
    offs = (-40, -2, -1, 0, 1, 2, 40)
    rows = np.concatenate([r[(r + d >= 0) & (r + d < m)] for d in offs])
    cols = np.concatenate([r[(r + d >= 0) & (r + d < m)] + d for d in offs])
    vals = rng.uniform(-1, 1, len(rows)) * 10.0 ** rng.integers(-8, 8, len(rows))
    x = rng.uniform(-1, 1, m) * 10.0 ** rng.integers(-3, 3, m)
    return oracle.make_coo(rows, cols, vals), m, m, x


@pytest.mark.gpu
@pytest.mark.parametrize("skew", ["0", "1"])
@pytest.mark.parametrize("relabel", ["0", "1"])
def test_every_finalize_path(eng, monkeypatch, skew, relabel):
    """Host and device multiply, y = alpha A x + beta y, the dot pass and a diag_limit pass, on either walk, with and
    without relabelled rows"""
    import torch

    monkeypatch.setenv("SMVP_TJDS_SKEW", skew)
    monkeypatch.setenv("SMVP_TJDS_RELABEL", relabel)
    coo, m, n, x = band_data()
    A = eng.TjdsMatrix.build(coo, m, n)
    rng = np.random.default_rng(41)
    perm, sp, ri, va = A.export()
    lim = A.ndiag // 2
    walked = oracle.make_coo(ri[:sp[lim]], perm[np.arange(sp[lim]) - np.repeat(sp[:lim], np.diff(sp[:lim + 1]))],
                             va[:sp[lim]])
    dx = _cuda(x)
    for v in (DET, FAST):
        want = model(coo, m, x, v)
        y, _ = A.mult(x, 1, v)
        same_bits(y, want, "host")
        A.set_x_device(dx)
        dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
        A.mult_device(dy, v)
        same_bits(dy.cpu().numpy(), want, "device")
        for alpha, beta in ((1.0, 0.0), (-0.75, 1.0), (2.5, -1.25)):
            y0 = rng.uniform(-2, 2, m)
            exp = alpha * want if beta == 0.0 else alpha * want + beta * y0
            dy = _cuda(y0)
            A.mult_device_axpby(alpha, beta, dy, v)
            same_bits(dy.cpu().numpy(), exp, "axpby %r %r" % (alpha, beta))
            dy, dd = _cuda(y0), torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
            A.mult_device_axpby_dot(alpha, beta, dy, None, dd, v)
            same_bits(dy.cpu().numpy(), exp, "dot %r %r" % (alpha, beta))
            # w = y_new: the terms are >= 0, the fixed-order sum is within a few dozen roundings of the exact one
            dot, ref = dd.cpu().numpy()[0], math.fsum((exp * exp).tolist())
            assert abs(dot - ref) <= 64 * 2.0 ** -53 * ref, (dot, ref)
            dy2, dd2 = _cuda(y0), torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
            A.mult_device_axpby_dot(alpha, beta, dy2, None, dd2, v)
            assert util_bits(dd2.cpu().numpy()[0]) == util_bits(dot)
        dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
        A.mult_device(dy, v, lim)
        same_bits(dy.cpu().numpy(), model(coo, m, x, v, walked), "diag_limit %d" % lim)
        assert A.plan()[1] == 1
    assert A.plan()[0] == (1 if skew == "1" else -1)
    assert A.y_relabel == (1 if relabel == "1" else -1)
    A.free()


@pytest.mark.gpu
def test_device_built_stencil(eng):
    """48^3 27-point stencil with hashed values, built on the device, against the numpy model (2.9 M entries)"""
    import torch

    nx = 48
    m = n = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=3)
    coo = oracle.make_coo(torch.as_tensor(r, device="cuda").cpu().numpy(), torch.as_tensor(c, device="cuda").cpu().numpy(),
                          torch.as_tensor(v, device="cuda").cpu().numpy())
    x = synth_ref.vector(n, 77)
    want = model_np(coo, m, x)
    T = eng.TjdsMatrix.build_device(r, c, v, m, n, r.n)
    T.set_x_device(_cuda(x))
    for variant in (DET, FAST):
        dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
        T.mult_device(dy, variant)
        same_bits(dy.cpu().numpy(), want[variant], "variant %d" % variant)
        assert T.plan()[1] == 1
    T.free()
