"""The reductions behind the heat map (recoup_b200/csrc/consumers.cu) against exact references:
rcp_matrix_row_stat, rcp_order, rcp_matrix_quantile, rcp_reads_width_quantile and the non-finite
part of the column profiles.

References, all in this file and all exact:
  * row sum   math.fsum (the correctly rounded exact sum), bit for bit;
  * row mean  float(Fraction(exact sum) / n), bit for bit;
  * row max   the maximum, NaN when a cell is NaN;
  * order     a stable argsort with NaN dropped (O.r_sort_index), index for index;
  * quantile  R's quantile.default type 7 on a numpy sort: index <- 1 + (n - 1) * p,
              lo <- floor(index), h <- index - lo, (1 - h) * x[lo] + h * x[hi], every operation
              rounded on its own (no FMA), bit for bit.
Sums and means are compared bit for bit on realistic rows (gamma cells with zeros, counts, bin
means k / w, one-decimal values with negatives and -0.0, values spread over +-20 decades): the
kernel carries them as double-double (Ogita-Rump-Oishi Sum2), and a plain double sum differs from
the exact sum in most of these rows.  On a pathological family (+-1e16 and +-2^60 cancelling
among +-1, +-3, +-1e-3) only Sum2's bound holds: |sum - S| <= eps |S| + gamma_{n-1}^2 sum|x|, eps = 2^-53.

Non-finite rule of row sums and means (and of the column means of colProfile):
  * NaN if a cell is NaN or the row holds both +Inf and -Inf;
  * otherwise +-Inf if a cell is infinite;
  * a finite row whose running double sum overflows gives that infinity, never NaN.  R's
    long-double accumulator can return a finite value there.
-0.0 and +0.0 compare equal in every bit-for-bit check (the kernels key them alike).

The pure-host tests restate the kernels' arithmetic and show that these inputs tell a right
kernel from a wrong one.  Run the GPU tests with `-m gpu` on a B200."""
import ctypes as C
import functools
import math
import zlib
from fractions import Fraction

import numpy as np
import pytest

from oracle import recoup_oracle as O

EPS = 2.0 ** -53
DBL_MAX = np.finfo(np.float64).max
INF = float("inf")
NAN = float("nan")
FAMILIES = ["gamma", "counts", "bin_means", "decimal", "decades"]
BIN_WIDTHS = np.array([25.0, 37.0, 50.0, 100.0, 133.0])
ROW_SHAPES = [(1, 1), (1, 2000), (255, 37), (256, 200), (257, 1), (257, 2), (257, 37), (257, 200), (257, 2000),
              (65537, 37), (1_000_000, 2)]
LADDER = (0.95, 0.96, 0.97, 0.98, 0.99, 0.995, 0.999)          # heatmapScale's probabilities
ORDER_N = [1, 2, 3, 255, 256, 257, (1 << 16) - 1, (1 << 16) + 1, 300001, (1 << 22) + 5]
WHATS = ["sum1", "max1", "avg1", "suma", "maxa", "avga"]


def seed_of(*key):
    return zlib.crc32(repr(key).encode())


# ---- comparison ------------------------------------------------------------------------------
def bits(a):
    a = np.asarray(a, dtype=np.float64) + 0.0               # -0.0 -> +0.0
    b = a.view(np.int64).copy()
    b[np.isnan(a)] = -1
    return b


def assert_bits(got, want, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(bits(got) != bits(want))
    assert bad.size == 0, "%s: %d of %d differ, first at %d: got %r, want %r" % (
        what, bad.size, got.size, bad[0], got.flat[bad[0]], want.flat[bad[0]])


# ---- exact references ------------------------------------------------------------------------
def exact_sum(row):
    """the exact sum of a finite row, as a Fraction (common power-of-two denominator)"""
    pairs = [v.as_integer_ratio() for v in np.asarray(row, dtype=np.float64).tolist()]
    d = max(q for _, q in pairs)
    return Fraction(sum(p * (d // q) for p, q in pairs), d)


def _special(m):
    """rows whose sum is not finite under the rule, and that value"""
    with np.errstate(over="ignore", invalid="ignore"):
        run_end = np.cumsum(m, axis=1)
    rows = np.flatnonzero(~np.isfinite(run_end).all(axis=1) | ~np.isfinite(m).all(axis=1))
    val = {}
    for i in rows.tolist():
        r = m[i]
        pos, neg = bool(np.isposinf(r).any()), bool(np.isneginf(r).any())
        if np.isnan(r).any() or (pos and neg):
            val[i] = NAN
        elif pos or neg:
            val[i] = INF if pos else -INF
        else:                                                # a finite row: the first overflow
            with np.errstate(over="ignore"):
                run = np.cumsum(r)
            val[i] = float(run[np.flatnonzero(~np.isfinite(run))[0]])
    return val


def ref_sum(m):
    m = np.asarray(m, dtype=np.float64)
    special = _special(m)
    out = np.empty(m.shape[0])
    for i, r in enumerate(m.tolist()):
        out[i] = special[i] if i in special else math.fsum(r)
    return out


def ref_mean(m, rows=None):
    m = np.asarray(m, dtype=np.float64)
    rows = range(m.shape[0]) if rows is None else rows
    special = _special(m)
    n = m.shape[1]
    return np.array([special[i] if i in special else float(exact_sum(m[i]) / n) for i in rows])


def ref_max(m):
    return np.asarray(m, dtype=np.float64).max(axis=1)     # NaN propagates


def ref_row_stat(m, kind):
    return {"sum": ref_sum, "avg": ref_mean, "max": ref_max}[kind](m)


def r_quantile7(x, probs):
    """quantile.default type 7, operation for operation (the oracle restates the same)"""
    return O.r_quantile7(x, probs)


def q7_old_index(x, probs):
    """the former form: index = (n - 1) p, h = index - floor(index), 0-based reads"""
    xs = np.sort(np.asarray(x, dtype=np.float64).ravel())
    out = []
    for p in probs:
        index = (xs.size - 1) * float(p)
        lo, hi = math.floor(index), math.ceil(index)
        h = index - lo
        q = xs[lo]
        if index > lo and xs[hi] != q:
            q = (1.0 - h) * q + h * xs[hi]
        out.append(float(q))
    return np.array(out)


def q7_fma(x, probs):
    """R's index, but the interpolation contracted into one FMA: fma(h, x[hi], (1 - h) x[lo])"""
    xs = np.sort(np.asarray(x, dtype=np.float64).ravel())
    out = []
    for p in probs:
        index = 1.0 + (xs.size - 1) * float(p)
        lo, hi = math.floor(index), math.ceil(index)
        h = index - lo
        q = float(xs[lo - 1])
        xh = float(xs[hi - 1])
        if index > lo and xh != q and math.isfinite(q) and math.isfinite(xh):
            q = float(Fraction(h) * Fraction(xh) + Fraction((1.0 - h) * q))
        out.append(q)
    return np.array(out)


# ---- restatements of the kernel's arithmetic (host tests) -----------------------------------
def dd_rows(m):
    """row_stat_kernel's sum: TwoSum per column, in column order, every row at once; the error
    term is dropped once the plain sum is not finite"""
    m = np.asarray(m, dtype=np.float64)
    hi, lo = np.zeros(m.shape[0]), np.zeros(m.shape[0])
    with np.errstate(over="ignore", invalid="ignore"):
        for c in range(m.shape[1]):
            x = m[:, c]
            s = hi + x
            bb = s - hi
            err = (hi - (s - bb)) + (x - bb)
            lo = np.where(np.isfinite(s), lo + err, 0.0)
            hi = s
    return hi, lo


def dd_sum(m):
    hi, lo = dd_rows(m)
    with np.errstate(invalid="ignore"):
        return hi + lo


def dd_mean(m, rows=None):
    """dd_div: q = s / n, r = fma(-q, n, s) + rest, q + r / n (the FMA exact, via Fraction)"""
    hi, lo = dd_rows(m)
    n = float(m.shape[1])
    out = []
    for i in (range(m.shape[0]) if rows is None else rows):
        s = hi[i] + lo[i]
        q = s / n
        if not math.isfinite(s):
            out.append(q)
            continue
        rest = (hi[i] - s) + lo[i]
        r = float(Fraction(-q) * Fraction(n) + Fraction(s)) + rest
        out.append(q + r / n)
    return np.array(out)


def naive_sum(m):
    m = np.asarray(m, dtype=np.float64)
    s = np.zeros(m.shape[0])
    with np.errstate(over="ignore", invalid="ignore"):
        for c in range(m.shape[1]):
            s = s + m[:, c]
    return s


def naive_row_stat(m, kind):
    if kind == "max":
        return ref_max(m)
    s = naive_sum(m)
    return s if kind == "sum" else s / m.shape[1]


# ---- inputs ----------------------------------------------------------------------------------
def family(name, rng, n_rows, n_cols):
    shape = (n_rows, n_cols)
    if name == "gamma":
        a = rng.gamma(0.6, 3.0, size=shape)
        a[rng.random(shape) < 0.3] = 0.0
    elif name == "counts":
        a = rng.poisson(4.0, size=shape).astype(np.float64)
    elif name == "bin_means":
        a = rng.integers(0, 4000, size=shape) / rng.choice(BIN_WIDTHS, size=n_cols)[None, :]
    elif name == "decimal":
        a = np.round(rng.normal(0.0, 2.0, size=shape), 1)
        a[rng.random(shape) < 0.05] = -0.0
    elif name == "decades":
        a = rng.choice([-1.0, 1.0], size=shape) * 10.0 ** rng.uniform(-20.0, 20.0, size=shape)
    else:
        raise ValueError(name)
    return np.asfortranarray(a)


def mean_rows(n_rows, rng):
    """every row of a small matrix; else 2 000 seeded rows plus both sides of every 256-row boundary"""
    if n_rows <= 4096:
        return np.arange(n_rows)
    edge = np.flatnonzero((np.arange(n_rows) % 256 == 0) | (np.arange(n_rows) % 256 == 255))
    return np.union1d(np.union1d(rng.choice(n_rows, 2000, replace=False), edge), [n_rows - 1])


@functools.lru_cache(maxsize=None)
def row_case(name, n_rows, n_cols):
    rng = np.random.default_rng(seed_of(name, n_rows, n_cols))
    m = family(name, rng, n_rows, n_cols)
    rows = mean_rows(n_rows, rng)
    return m, ref_sum(m), rows, ref_mean(m, rows), ref_max(m)


def pathological(n_rows, n_cols, seed):
    """rows of +-1e16 and +-2^60 that cancel exactly, among small cells +-1, +-3, +-1e-3, shuffled:
    the exact sum is small next to sum|x|, so a plain double sum loses it"""
    rng = np.random.default_rng(seed)
    m = np.empty((n_rows, n_cols))
    for i in range(n_rows):
        k = int(rng.integers(1, n_cols // 4 + 1))
        j = int(rng.integers(0, k + 1))
        big = [1e16, -1e16] * (k - j) + [2.0 ** 60, -2.0 ** 60] * j
        small = rng.choice([1.0, 3.0, 1e-3, -1.0, -3.0, -1e-3], size=n_cols - 2 * k)
        m[i] = rng.permutation(np.concatenate([big, small]))
    return np.asfortranarray(m)


def sum2_bound_ok(got, row):
    """|got - S| <= eps |S| + gamma_{n-1}^2 sum|x|, in exact arithmetic; returns (ok, error / bound)"""
    S = exact_sum(row)
    k = Fraction(row.shape[0] - 1)
    e = Fraction(EPS)
    gamma = k * e / (1 - k * e)
    bound = e * abs(S) + gamma * gamma * exact_sum(np.abs(row))
    err = abs(Fraction(got) - S)
    return err <= bound, (float(err / bound) if bound else float(err != 0))


def near_tie_pairs(n_pairs, n_cols, seed):
    """(B, A) row pairs of bin means: B is a column permutation of A with one cell raised by one
    ulp of A's sum, so the exact sums (and means) round one ulp apart, B above A, while the plain
    double sum and mean put B strictly below A."""
    rng = np.random.default_rng(seed)
    n = float(n_cols)
    out = []
    while len(out) < n_pairs:
        a = rng.integers(0, 4000, size=n_cols) / rng.choice(BIN_WIDTHS, size=n_cols)
        S = exact_sum(a)
        s = float(S)
        u = float(np.spacing(s))
        j = int(np.argmax(a))
        if Fraction(a[j]) + Fraction(u) != Fraction(a[j] + u):
            continue
        b = a.copy()
        b[j] += u
        if math.fsum(b) != np.nextafter(s, INF) or not float((S + Fraction(u)) / n) > float(S / n):
            continue
        cand = b[np.array([rng.permutation(n_cols) for _ in range(64)])]
        na = naive_sum(a[None, :])[0]
        nb = naive_sum(cand)
        ok = np.flatnonzero((nb < na) & (nb / n < na / n))
        if ok.size:
            out.append((cand[ok[0]], a))
    return out


@functools.lru_cache(maxsize=1)
def order_matrix():
    """near-tie pairs, groups of rows that are column permutations of each other, a +Inf row,
    a -Inf row and a row with both; returns (matrix, rows of those three, 0-based)"""
    n_cols = 200
    rng = np.random.default_rng(seed_of("order_matrix"))
    rows = [r for pair in near_tie_pairs(24, n_cols, seed_of("pairs")) for r in pair]
    for _ in range(4):
        base = family("gamma", rng, 1, n_cols)[0]
        rows += [base[rng.permutation(n_cols)] for _ in range(5)]
    plus = family("gamma", rng, 1, n_cols)[0]
    plus[17] = INF
    minus = np.full(n_cols, -INF)
    both = family("gamma", rng, 1, n_cols)[0]
    both[3], both[150] = INF, -INF
    at = len(rows) // 2
    rows[at:at] = [plus, minus, both]
    return np.asfortranarray(np.array(rows)), (at, at + 1, at + 2)


def order_input(what):
    m, _ = order_matrix()
    return [{"profile": m}, {"profile": np.asfortranarray(m.copy())}] if what.endswith("a") else [{"profile": m}]


def order_values(inp, what, stat):
    kind = what[:3]
    if what.endswith("a"):
        per = np.stack([stat(x["profile"], kind) for x in inp], axis=1)
        return stat(per, kind)
    return stat(inp[0]["profile"], kind)


def order_values_of(k, n, rng):
    """n values of kind k (ORDER_KINDS)"""
    if k == "ties":
        return rng.integers(0, 4, size=n).astype(np.float64)
    if k == "equal":
        return np.full(n, 2.5)
    if k == "zeros":
        return rng.choice([0.0, -0.0], size=n)
    if k == "extremes":
        return rng.choice([0.0, -0.0, 5e-324, -5e-324, DBL_MAX, -DBL_MAX, INF, -INF, 1.0], size=n)
    if k == "rounded":
        return np.round(rng.normal(size=n), 2)
    v = order_values_of("extremes" if k == "nan_half" else "ties", n, rng)
    if k == "nan_first":
        v[0] = NAN
    elif k == "nan_last":
        v[-1] = NAN
    elif k == "nan_half":
        v[rng.random(n) < 0.5] = NAN
    elif k == "nan_all":
        v[:] = NAN
    return v


ORDER_KINDS = ["ties", "equal", "zeros", "extremes", "rounded", "nan_first", "nan_last", "nan_half", "nan_all"]


def quantile_probs(n):
    """0, 1, 0.1, the ladder, k / (n - 1) in double for a few k, and nextafter on both sides"""
    ps = [0.0, 1.0, 0.1, 0.25, 0.5] + list(LADDER)
    if n > 2:
        ps += [k / (n - 1) for k in sorted({1, 2, n // 3, n // 2, n - 2})]
    out = []
    for p in ps:
        out += [p, np.nextafter(p, 0.0), np.nextafter(p, 1.0)]
    return np.array(sorted(set(out)))


def quantile_matrix(kind, n_rows, n_cols, rng):
    shape = (n_rows, n_cols)
    if kind == "sparse":                                     # mostly zeros
        a = np.zeros(shape)
        hit = rng.random(shape) < 0.02
        a[hit] = rng.gamma(0.6, 3.0, size=int(hit.sum()))
    elif kind == "ties":
        a = rng.integers(0, 5, size=shape).astype(np.float64)
    elif kind == "negative":
        a = np.round(rng.normal(0.0, 2.0, size=shape), 1)
    elif kind == "inf":
        a = rng.gamma(0.6, 3.0, size=shape)
        a[rng.random(shape) < 0.1] = INF
        a[rng.random(shape) < 0.1] = -INF
    else:
        a = rng.gamma(0.6, 3.0, size=shape)
    return np.asfortranarray(a)


QUANTILE_SHAPES = [(1, 1), (2, 1), (1, 3), (5, 2), (101, 1), (20000, 200), ((1 << 24) + 3, 1)]
QUANTILE_KINDS = ["gamma", "sparse", "ties", "negative", "inf"]


def quantile_cases(n_rows, n_cols):
    rng = np.random.default_rng(seed_of("quantile", n_rows, n_cols))
    big = n_rows * n_cols > 1_000_000
    for kind in (["sparse", "inf"] if big else QUANTILE_KINDS):
        yield kind, quantile_matrix(kind, n_rows, n_cols, rng)
    if n_rows * n_cols == 2:
        yield "zero_one", np.asfortranarray([[0.0], [1.0]])


# ------------------------------------------------------------------------------ host tests --
@pytest.mark.parametrize("shape", ROW_SHAPES, ids=lambda s: "%dx%d" % s)
def test_double_double_restatement_is_exact_on_every_realistic_row(shape):
    for name in FAMILIES:
        m, want_sum, rows, want_mean, _ = row_case(name, *shape)
        assert_bits(dd_sum(m), want_sum, "%s sum" % name)
        assert_bits(dd_mean(m, rows), want_mean, "%s mean" % name)


def test_plain_double_sum_differs_from_the_exact_sum_on_realistic_rows():
    """a kernel that sums in plain doubles would fail the bit-for-bit comparisons above"""
    for name in ["gamma", "bin_means", "decimal"]:
        m, want_sum, _, _, _ = row_case(name, 257, 200)
        assert (bits(naive_sum(m)) != bits(want_sum)).mean() > 0.3, name


@pytest.mark.parametrize("what", WHATS)
def test_plain_double_sum_fails_the_near_tie_order(what):
    m, (plus, minus, both) = order_matrix()
    inp = order_input(what)
    for dec in (False, True):
        want = O.r_sort_index(order_values(inp, what, ref_row_stat), dec)
        restated = O.r_sort_index(order_values(inp, what, lambda x, k: dd_mean(x) if k == "avg" else
                                                (dd_sum(x) if k == "sum" else ref_max(x))), dec)
        assert np.array_equal(restated, want)
        naive = O.r_sort_index(order_values(inp, what, naive_row_stat), dec)
        if what[:3] == "max":
            assert np.array_equal(naive, want)               # max is exact either way
        else:
            assert not np.array_equal(naive, want)
            assert both + 1 not in want and want.shape[0] == m.shape[0] - 1


def test_sum2_bound_holds_on_the_pathological_family():
    for n_cols in (37, 200, 2000):
        m = pathological(100, n_cols, seed_of("pathological", n_cols))
        got, naive = dd_sum(m), naive_sum(m)
        naive_out = 0
        for i in range(m.shape[0]):
            ok, ratio = sum2_bound_ok(got[i], m[i])
            assert ok, (n_cols, i, ratio)
            naive_out += not sum2_bound_ok(naive[i], m[i])[0]
        # pathological: the plain sum leaves the bound, and Sum2 is not always correctly rounded here
        assert naive_out > 90 and (bits(got) != bits(ref_sum(m))).any(), n_cols


def test_quantile_index_forms_differ_on_the_chosen_probabilities():
    """R's index = 1 + (n - 1) p, and separately rounded products, against the (n - 1) p form and an
    FMA-contracted interpolation: both differ somewhere on the inputs the GPU tests use"""
    assert r_quantile7([0.0, 1.0], [0.1])[0] == 0.10000000000000009
    assert q7_old_index([0.0, 1.0], [0.1])[0] == 0.1
    old_diff = fma_diff = total = 0
    for shape in QUANTILE_SHAPES[:-2]:
        for _, m in quantile_cases(*shape):
            p = quantile_probs(m.size)
            want = r_quantile7(m, p)
            old_diff += int((bits(q7_old_index(m, p)) != bits(want)).sum())
            fma_diff += int((bits(q7_fma(m, p)) != bits(want)).sum())
            total += p.size
    assert old_diff > 0 and fma_diff > 0, (old_diff, fma_diff, total)


def test_known_quantiles_of_r():
    assert r_quantile7([5.0], [0.0, 0.3, 1.0]).tolist() == [5.0, 5.0, 5.0]
    assert r_quantile7([-INF, 1.0, INF], [0.25, 0.5, 0.75]).tolist() == [-INF, 1.0, INF]


# ------------------------------------------------------------------------------- GPU tests --
@pytest.fixture(scope="session")
def rb():
    import recoup_b200 as rb
    rb.init(0)
    return rb


def _lib():
    from recoup_b200 import _lib as L
    return L


def _vp(a):
    return C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())


def to_device(a):
    """a numpy array as a CUDA tensor with the same (column-major) layout"""
    import torch
    a = np.asarray(a)
    if a.ndim == 2:
        return torch.from_numpy(np.ascontiguousarray(np.asfortranarray(a).T)).cuda()
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def row_stat(m, what, mem="host", n_rows=None, ld=None, offset=0):
    L = _lib()
    code = {"sum": 0, "max": 1, "avg": 2}[what]
    m = np.asfortranarray(m)
    n_rows = m.shape[0] if n_rows is None else n_rows
    ld = m.shape[0] if ld is None else ld
    if mem == "host":
        out = np.full(n_rows, 7.0)
        L.check(L.lib.rcp_matrix_row_stat(C.c_void_p(m.ctypes.data + 8 * offset), n_rows, m.shape[1], ld, code,
                                          L.MEM_HOST, _vp(out)))
        return out
    import torch
    dm = to_device(m)
    out = torch.full((n_rows,), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    L.check(L.lib.rcp_matrix_row_stat(C.c_void_p(dm.data_ptr() + 8 * offset), n_rows, m.shape[1], ld, code,
                                      L.MEM_DEVICE, _vp(out)))
    L.check(L.lib.rcp_sync())
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ROW_SHAPES, ids=lambda s: "%dx%d" % s)
def test_row_stat_exact(rb, shape):
    for name in FAMILIES:
        m, want_sum, rows, want_mean, want_max = row_case(name, *shape)
        mem = "device" if name in ("gamma", "decades") else "host"
        assert_bits(row_stat(m, "sum", mem), want_sum, "%s %s sum" % (name, mem))
        assert_bits(row_stat(m, "avg", mem)[rows], want_mean, "%s %s mean" % (name, mem))
        assert_bits(row_stat(m, "max", mem), want_max, "%s %s max" % (name, mem))


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
def test_row_stat_of_a_row_block(rb, mem):
    """rows [r0, r0 + n) of a wider matrix: leading dimension > n_rows, straight through the C ABI"""
    m, _, _, _, _ = row_case("bin_means", 65537, 37)
    for r0, n in [(0, 1), (0, 300), (1, 256), (255, 257), (1000, 60000)]:
        block = m[r0:r0 + n]
        for what, ref in [("sum", ref_sum), ("avg", ref_mean), ("max", ref_max)]:
            got = row_stat(m, what, mem, n_rows=n, ld=m.shape[0], offset=r0)
            if what == "avg" and n > 4096:
                rows = np.arange(0, n, 97)
                assert_bits(got[rows], ref_mean(block, rows), "block %d+%d mean" % (r0, n))
            else:
                assert_bits(got, ref(block), "block %d+%d %s" % (r0, n, what))


@pytest.mark.gpu
def test_row_stat_sum2_bound_on_the_pathological_family(rb):
    for n_cols, mem in [(37, "host"), (200, "device"), (2000, "host")]:
        m = pathological(1000 if n_cols < 2000 else 100, n_cols, seed_of("pathological device", n_cols))
        got = row_stat(m, "sum", mem)
        for i in range(m.shape[0]):
            ok, ratio = sum2_bound_ok(got[i], m[i])
            assert ok, (n_cols, i, ratio)


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
def test_row_stat_non_finite(rb, mem):
    rows = [
        [1.0, INF, 2.0],                         # +Inf
        [0.5, -INF],                             # -Inf
        [-INF, -INF, 3.0],
        [INF, -INF, 1.0],                        # both: NaN
        [1.0, NAN, 2.0],                         # NaN
        [NAN, INF, 1.0],
        [1.7e308, 1.7e308, -1.7e308],            # finite, the running sum overflows: +Inf
        [-1.7e308, -1.7e308, 1.0],               # -Inf
        [DBL_MAX, -DBL_MAX, DBL_MAX],            # finite, no overflow
        [5e-324, 5e-324, -5e-324],
        [-0.0, -0.0, -0.0],
    ]
    width = max(len(r) for r in rows)
    # pad every row to one width with zeros, which change no sum; the mean divides by the width
    m = np.asfortranarray([r + [0.0] * (width - len(r)) for r in rows])
    want_sum = ref_sum(m)
    assert want_sum[:3].tolist() == [INF, -INF, -INF] and np.isnan(want_sum[3:6]).all()
    assert want_sum[6:9].tolist() == [INF, -INF, DBL_MAX]
    assert_bits(row_stat(m, "sum", mem), want_sum, "sum")
    assert_bits(row_stat(m, "avg", mem), ref_mean(m), "mean")
    assert_bits(row_stat(m, "max", mem), ref_max(m), "max")
    for r in rows:                                       # unpadded: mean(0.5, -Inf) = -Inf
        one = np.asfortranarray([r])
        assert_bits(row_stat(one, "sum", mem), ref_sum(one), repr(r))
        assert_bits(row_stat(one, "avg", mem), ref_mean(one), repr(r))


@pytest.mark.gpu
def test_row_stat_errors(rb):
    L = _lib()
    m = np.asfortranarray(np.ones((4, 3)))
    out = np.empty(4)
    assert L.lib.rcp_matrix_row_stat(_vp(m), 4, 0, 4, 0, L.MEM_HOST, _vp(out)) == L.RCP_ERR_ARG
    for bad in (-1, 3):
        assert L.lib.rcp_matrix_row_stat(_vp(m), 4, 3, 4, bad, L.MEM_HOST, _vp(out)) == L.RCP_ERR_ARG
    assert L.lib.rcp_matrix_row_stat(_vp(m), 4, 3, 4, 0, L.MEM_HOST, None) == L.RCP_ERR_ARG
    assert L.lib.rcp_matrix_row_stat(_vp(m), 4, 3, 3, 0, L.MEM_HOST, _vp(out)) == L.RCP_ERR_ARG      # ld < rows
    assert L.lib.rcp_matrix_row_stat(_vp(m), 0, 3, 1, 0, L.MEM_HOST, _vp(out)) == L.RCP_OK           # no rows


def order(v, dec, mem="host", with_n_out=True):
    L = _lib()
    v = np.ascontiguousarray(v, dtype=np.float64)
    n_out = C.c_int64(-1)
    n_ptr = C.byref(n_out) if with_n_out else None
    if mem == "host":
        ix = np.zeros(v.shape[0], dtype=np.int32)
        L.check(L.lib.rcp_order(_vp(v), v.shape[0], int(dec), L.MEM_HOST, _vp(ix), n_ptr))
    else:
        import torch
        dv = to_device(v)
        dix = torch.zeros(v.shape[0], dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        L.check(L.lib.rcp_order(_vp(dv), v.shape[0], int(dec), L.MEM_DEVICE, _vp(dix), n_ptr))
        ix = dix.cpu().numpy()
    return ix, (n_out.value if with_n_out else None)


@pytest.mark.gpu
@pytest.mark.parametrize("n", ORDER_N)
def test_order_equals_a_stable_argsort(rb, n):
    rng = np.random.default_rng(seed_of("order", n))
    for j, kind in enumerate(ORDER_KINDS):
        v = order_values_of(kind, n, rng)
        n_valid = int((~np.isnan(v)).sum())
        for dec in (False, True):
            want = O.r_sort_index(v, dec)
            mem = "device" if (j + dec) % 3 == 0 else "host"
            ix, n_out = order(v, dec, mem, with_n_out=(j + dec) % 4 != 1)
            if n_out is not None:
                assert n_out == n_valid, (kind, dec, mem)
            assert np.array_equal(ix[:n_valid], want), (kind, dec, mem)


@pytest.mark.gpu
@pytest.mark.parametrize("order_", ["ascending", "descending"])
@pytest.mark.parametrize("what", WHATS)
def test_order_profiles_exact(rb, what, order_):
    """exact ties keep input order both ways, one-ulp pairs come out in exact order, +-Inf rows
    stay at the ends and an Inf/-Inf row is dropped"""
    m, (plus, minus, both) = order_matrix()
    inp = order_input(what)
    dec = order_ == "descending"
    val = order_values(inp, what, ref_row_stat)
    want = O.r_sort_index(val, dec)
    got = rb.orderProfiles(inp, {"orderBy": {"what": what, "order": order_}})["ix"]
    assert np.array_equal(got, want)
    assert_bits(rb.rowStat(m, what[:3]), ref_row_stat(m, what[:3]), what)
    if what[:3] != "max":
        assert got.shape[0] == m.shape[0] - 1 and both + 1 not in got
        first, last = (plus, minus) if dec else (minus, plus)
        assert got[0] == first + 1 and got[-1] == last + 1


def matrix_quantile(m, probs, mem="host", n_rows=None, ld=None, offset=0):
    L = _lib()
    m = np.asfortranarray(m)
    p = np.ascontiguousarray(probs, dtype=np.float64)
    out = np.full(p.shape[0], 7.0)
    n_rows = m.shape[0] if n_rows is None else n_rows
    ld = m.shape[0] if ld is None else ld
    if mem == "host":
        L.check(L.lib.rcp_matrix_quantile(C.c_void_p(m.ctypes.data + 8 * offset), n_rows, m.shape[1], ld, _vp(p),
                                          p.shape[0], L.MEM_HOST, _vp(out)))
    else:
        import torch
        dm = to_device(m)
        torch.cuda.synchronize()
        L.check(L.lib.rcp_matrix_quantile(C.c_void_p(dm.data_ptr() + 8 * offset), n_rows, m.shape[1], ld,
                                          _vp(p), p.shape[0], L.MEM_DEVICE, _vp(out)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape", QUANTILE_SHAPES, ids=lambda s: "%dx%d" % s)
def test_matrix_quantile_exact(rb, shape):
    for j, (kind, m) in enumerate(quantile_cases(*shape)):
        p = quantile_probs(m.size)
        mem = "device" if j % 2 else "host"
        assert_bits(matrix_quantile(m, p, mem), r_quantile7(m, p), "%s %s" % (kind, mem))


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
def test_matrix_quantile_of_a_row_block(rb, mem):
    rng = np.random.default_rng(seed_of("quantile block"))
    m = quantile_matrix("ties", 1000, 7, rng)
    m[:, 3] = rng.normal(size=1000)
    for r0, n in [(0, 1), (3, 10), (100, 257)]:
        block = m[r0:r0 + n]
        p = quantile_probs(block.size)
        assert_bits(matrix_quantile(m, p, mem, n_rows=n, ld=m.shape[0], offset=r0), r_quantile7(block, p),
                    "block %d+%d" % (r0, n))


@pytest.mark.gpu
def test_matrix_quantile_errors(rb):
    L = _lib()
    m = np.asfortranarray(np.arange(12.0).reshape(4, 3))
    out = np.empty(1)

    def call(mat, probs, k=None):
        p = np.ascontiguousarray(probs, dtype=np.float64)
        return L.lib.rcp_matrix_quantile(_vp(mat), mat.shape[0], mat.shape[1], mat.shape[0], _vp(p),
                                         p.shape[0] if k is None else k, L.MEM_HOST, _vp(out))
    bad = m.copy(order="F")
    bad[2, 1] = NAN
    assert call(bad, [0.5]) == L.RCP_ERR_DATA
    for p in (NAN, -1e-300, -0.5, 1.0000000000000002, 2.0, INF):
        assert call(m, [p]) == L.RCP_ERR_ARG, p
    assert call(m, [0.5, NAN]) == L.RCP_ERR_ARG
    assert call(m, [0.5], k=0) == L.RCP_OK
    assert L.lib.rcp_matrix_quantile(_vp(m), 4, 3, 4, None, 0, L.MEM_HOST, None) == L.RCP_OK
    assert call(m, [0.5], k=-1) == L.RCP_ERR_ARG
    assert call(m, [-0.0]) == L.RCP_OK and out[0] == 0.0


@pytest.mark.gpu
def test_heatmap_scale(rb):
    rng = np.random.default_rng(seed_of("heatmap"))
    a = quantile_matrix("gamma", 2001, 37, rng)
    b = quantile_matrix("sparse", 500, 37, rng)
    zero = np.zeros((300, 37))
    inp = [{"profile": a}, {"profile": b}, {"profile": zero}]
    for factor in (1.0, 0.5, 3.0):
        got = rb.heatmapScale(inp, "each", factor)
        for g, x in zip(got, inp):
            nz = [q for q in r_quantile7(x["profile"], LADDER) if q != 0]
            assert_bits([g], [factor * (nz[0] if nz else 0.0)])
        assert got[2] == 0.0
        sup = max(float(r_quantile7(x["profile"], [0.95])[0]) for x in inp)
        assert_bits(rb.heatmapScale(inp, "common", factor), [factor * sup] * 3)
    # the 0.95 .. 0.99 quantiles of `sparse` are 0: "each" climbs the ladder
    sparse = np.zeros((100, 10))
    sparse[0, :3] = [4.0, 5.0, 6.0]
    want = [q for q in r_quantile7(sparse, LADDER) if q != 0][0]
    assert_bits(rb.heatmapScale([{"profile": sparse}], "each"), [want])


def width_quantile(start, end, prob, mem="host"):
    L = _lib()
    s = np.ascontiguousarray(start, dtype=np.int32)
    e = np.ascontiguousarray(end, dtype=np.int32)
    q, n_le = C.c_double(-1.0), C.c_int64(-1)
    if mem == "host":
        L.check(L.lib.rcp_reads_width_quantile(s.shape[0], _vp(s), _vp(e), float(prob), L.MEM_HOST,
                                               C.byref(q), C.byref(n_le)))
    else:
        import torch
        ds, de = to_device(s), to_device(e)
        torch.cuda.synchronize()
        L.check(L.lib.rcp_reads_width_quantile(s.shape[0], _vp(ds), _vp(de), float(prob), L.MEM_DEVICE,
                                               C.byref(q), C.byref(n_le)))
    return q.value, n_le.value


def width_cases():
    rng = np.random.default_rng(seed_of("widths"))
    yield "one", np.array([100]), np.array([150])
    yield "equal", np.arange(1, 1001), np.arange(1, 1001) + 75
    s = rng.integers(1, 1000, size=5001)
    yield "mixed", s, s + rng.integers(0, 300, size=5001)
    s = np.ones(7, dtype=np.int64)
    yield "extremes", s, np.array([1, 1, 2147483647, 1, 2147483647, 50, 1])
    s = rng.integers(1, 10_000_000, size=300001)
    yield "large", s, s + rng.integers(0, 2000, size=300001)


@pytest.mark.gpu
def test_width_quantile_exact(rb):
    for j, (name, s, e) in enumerate(width_cases()):
        w = (e - s + 1).astype(np.float64)
        for p in (0.0, 0.75, 0.9, 1.0, 0.1, np.nextafter(0.75, 0.0), np.nextafter(0.75, 1.0), 1 / 3):
            want = float(r_quantile7(w, [p])[0])
            for mem in ("host", "device"):
                q, n_le = width_quantile(s, e, p, mem)
                assert_bits([q], [want], "%s p=%r %s" % (name, p, mem))
                assert n_le == int((~(w > want)).sum()), (name, p, mem)


@pytest.mark.gpu
def test_width_quantile_of_a_decoded_handle(rb):
    rng = np.random.default_rng(seed_of("bed"))
    cs = rng.integers(0, 1_000_000, size=2001)
    ce = cs + rng.integers(1, 400, size=2001)
    ce[:3] = cs[:3] + 1                                      # width 1
    text = "".join("chr1\t%d\t%d\n" % (a, b) for a, b in zip(cs, ce)).encode()
    gr = rb.readBed(text, ["chr1"], seqlengths=np.array([2_000_000], dtype=np.int64))
    assert gr.decoded_handle is not None
    w = (ce - cs).astype(np.float64)
    for p in (0.0, 0.75, 0.9, 1.0, 0.1, 1 / 3):
        want = float(r_quantile7(w, [p])[0])
        q, n_le = rb.widthQuantile(gr, p)
        assert_bits([q], [want], "p=%r" % p)
        assert n_le == int((~(w > want)).sum())


@pytest.mark.gpu
def test_width_quantile_errors(rb):
    L = _lib()
    s = np.ones(5, dtype=np.int32)
    e = np.arange(1, 6, dtype=np.int32)
    q, n_le = C.c_double(0.0), C.c_int64(0)
    for p in (NAN, -0.25, 1.5, -INF, INF):
        assert L.lib.rcp_reads_width_quantile(5, _vp(s), _vp(e), p, L.MEM_HOST, C.byref(q),
                                              C.byref(n_le)) == L.RCP_ERR_ARG, p
    gr = rb.readBed(b"chr1\t0\t5\nchr1\t3\t9\n", ["chr1"])
    for p in (NAN, 1.5):
        with pytest.raises(rb.RecoupError) as ei:
            rb.widthQuantile(gr, p)
        assert ei.value.code == L.RCP_ERR_ARG


def col_cases(scale):
    """columns: finite; +Inf; -Inf; +Inf and -Inf; -Inf, one finite cell and +Inf"""
    rng = np.random.default_rng(seed_of("col", scale))
    n = 41
    if scale == "log2":
        m = rng.choice([0.0, 1.0, 3.0, 7.0], size=(n, 5))
        m[6, 1] = INF
        m[9, 2] = -1.0                                       # log2(0) = -Inf
        m[4, 3], m[30, 3] = INF, -1.0
    else:
        m = np.round(rng.gamma(0.6, 3.0, size=(n, 5)), 2)
        m[6, 1] = INF
        m[9, 2] = -INF
        m[4, 3], m[30, 3] = INF, -INF
    m[:20, 4] = -INF if scale == "natural" else -1.0
    m[21:, 4] = INF
    return np.asfortranarray(m)


def scaled(x, scale):
    with np.errstate(divide="ignore"):
        return np.log2(x + 1.0) if scale == "log2" else x


def medians(x):
    with np.errstate(invalid="ignore"):                      # (-Inf + Inf) / 2 is NaN, as in R
        return [O.r_median(x[:, j]) for j in range(x.shape[1])]


def assert_col_stat(got, want, scale, what):
    """non-finite entries bit for bit; finite ones too on the natural scale.  Under log2 the
    device's log2 may differ from the host's in the last bit (even at powers of two), so finite
    entries there agree to a few ulps."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    fin = np.isfinite(want)
    if scale == "natural":
        assert_bits(got, want, what)
        return
    assert_bits(got[~fin], want[~fin], what)
    np.testing.assert_allclose(got[fin], want[fin], rtol=8 * EPS, atol=0, err_msg=what)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", ["natural", "log2"])
def test_col_profile_non_finite(rb, scale):
    m = col_cases(scale)
    center, spread = rb.colProfile(m, "mean", scale)
    assert center[1] == INF and np.isnan(spread[1])
    assert center[2] == -INF and np.isnan(spread[2])
    assert np.isnan(center[3]) and np.isnan(center[4])
    x = scaled(m, scale)
    assert_col_stat(center[:1], [float(exact_sum(x[:, 0]) / x.shape[0])], scale, "mean")
    med, _ = rb.colProfile(m, "median", scale)
    assert_col_stat(med, medians(x), scale, "median")
    # the same per group of rows (calcDesignPlotProfiles): every other row in group 2, row 0 excluded
    codes = (np.arange(m.shape[0]) % 2 + 1).astype(np.int32)
    codes[0] = 0
    gc, gs = rb.groupColProfile(m, codes, 2, "mean", scale)
    gm, _ = rb.groupColProfile(m, codes, 2, "median", scale)
    for g in (1, 2):
        xs = x[codes == g]
        s = ref_sum(xs.T)
        bad = ~np.isfinite(s)
        assert bad.sum() >= 2
        assert_bits(gc[g - 1, bad], s[bad] / xs.shape[0], "group %d mean" % g)
        assert np.isnan(gs[g - 1, bad]).all()
        assert_col_stat(gm[g - 1], medians(xs), scale, "group %d median" % g)
