"""Narrow (uint16) coverage storage of the split path: the same values as int32 storage
(RCP_COVERAGE_WIDE=1) and as the C oracle, the exact bound at 65 535 reads, and every reader of a
narrow handle.  Run with `-m gpu` on a B200."""
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import recoup_oracle as O
from tests.helpers import assert_coverage_equal, both_reads, both_regions, synth_reads

pytestmark = pytest.mark.gpu

LEVELS = ["a", "b", "c"]


@pytest.fixture
def rb():
    import recoup_b200 as rb
    rb.init(0)
    rb.set_coverage_path("split")
    yield rb
    rb.set_coverage_path("auto")


def storage_bytes(rb, cov):
    from recoup_b200 import _lib
    b = C.c_int(0)
    _lib.check(_lib.lib.rcp_coverage_storage_bytes(cov.handle, C.byref(b)))
    return b.value


def both_layouts(rb, monkeypatch, fn):
    """fn() under the default storage and under RCP_COVERAGE_WIDE=1."""
    monkeypatch.delenv("RCP_COVERAGE_WIDE", raising=False)
    narrow = fn()
    monkeypatch.setenv("RCP_COVERAGE_WIDE", "1")
    wide = fn()
    monkeypatch.delenv("RCP_COVERAGE_WIDE")
    return narrow, wide


def _shape(rng, kind, clen):
    """C2-like TSS windows or C3-like gene bodies (heavy-tailed lengths), reduced in scale."""
    R = 1500
    rc = rng.integers(0, 3, size=R)
    rst = rng.choice(np.array([1, -1], dtype=np.int8), size=R)
    if kind == "tss":
        tss = rng.integers(6000, 590_000, size=R)
        s2, e2 = O.get_regional_ranges(tss, tss, rst, "tss", (5000, 5000))
    else:
        gs = rng.integers(3000, 500_000, size=R)
        glen = np.minimum((rng.pareto(1.2, size=R) * 3000).astype(np.int64) + 50, 150_000)
        s2, e2 = O.get_regional_ranges(gs, gs + glen - 1, rst, "genebody", (2000, 2000))
    return rc, s2, e2, rst


@pytest.mark.parametrize("kind", ["tss", "genebody"])
def test_narrow_equals_wide_and_the_c_oracle(rb, monkeypatch, kind):
    rng = np.random.default_rng(501 if kind == "tss" else 502)
    clen = [3_000_000, 1_500_000, 700_000]
    chrom, s, e, st = synth_reads(rng, 600_000, clen, width=(200, 200))
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=LEVELS, seqlengths=clen)
    rc, s2, e2, rst = _shape(rng, kind, clen)
    g_mask = rb.GRanges(rc.astype(np.int32), s2, e2, strand=rst, seqlevels=LEVELS)
    dense = CO.coverage(CO.Index(chrom, s, e, st, clen), rc, s2, e2, rst)
    want = dense.to_list()

    def run():
        out = {}
        cov = rb.calcCoverage(g_reads, g_mask)
        out["bytes"] = storage_bytes(rb, cov)
        out["fetch"] = cov.to_list()
        out["rle"] = cov.rle(0, 300)
        for stat in ("mean", "median"):
            out["bins_" + stat] = np.asarray(rb.binCoverageMatrix(cov, binSize=100, stat=stat))
        # more bins than the 2000-base upstream segments have bases: the interpolation kernel
        for interp in ("spline", "neighborhood"):
            out["interp_" + interp] = np.asarray(rb.binCoverageMatrix(cov, binSize=2100, flank=(2000, 2000),
                                                                      where="upstream", interpolation=interp))
        out["bins_flank"] = np.asarray(rb.binCoverageMatrix(cov, binSize=40, flank=(2000, 2000), where="upstream"))
        out["base_up"] = np.asarray(rb.baseCoverageMatrix(cov, flank=(1000, 1000), where="upstream"))
        out["base_dn"] = np.asarray(rb.baseCoverageMatrix(cov, flank=(100, 37), where="downstream"))
        cov.set_scale(0.25)
        out["scaled"] = np.asarray(rb.binCoverageMatrix(cov, binSize=100))
        for filt in ("+", "-"):
            cf = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=False)
            out["strand" + filt] = (storage_bytes(rb, cf), cf.to_list(),
                                    np.asarray(rb.binCoverageMatrix(cf, binSize=100)))
        return out

    narrow, wide = both_layouts(rb, monkeypatch, run)
    assert narrow["bytes"] == 2 and wide["bytes"] == 4
    assert_coverage_equal(narrow["fetch"], want)
    for k in narrow:
        if k == "bytes":
            continue
        a, b = narrow[k], wide[k]
        if k == "fetch":
            assert_coverage_equal(a, [None if x is None else x.astype(np.int64) for x in b])
        elif k == "rle":
            assert len(a) == len(b)
            for x, y in zip(a, b):
                assert (x is None) == (y is None)
                if x is not None:
                    assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
        elif k.startswith("strand"):
            assert a[0] == 2 and b[0] == 4
            assert_coverage_equal(a[1], [None if x is None else x.astype(np.int64) for x in b[1]])
            assert np.array_equal(a[2], b[2], equal_nan=True), k
        else:
            assert np.array_equal(a, b, equal_nan=True), k
    assert np.array_equal(narrow["base_up"], O.base_coverage_matrix(want, (1000, 1000), "upstream"))


def _pileup(rb, n_pile, n_long=0):
    """n_pile identical 50-bp reads at 100 000 (plus n_long reads spanning it, kept out of the
    binned index) on a 400-kb chromosome; the background lies far beyond any tile's reach."""
    rng = np.random.default_rng(7)
    clen = [400_000]
    n_bg = 20_000
    s = np.concatenate([np.full(n_pile, 100_000), rng.integers(200_000, 390_000, size=n_bg),
                        np.full(n_long, 90_000)]).astype(np.int64)
    e = s + 49
    e[n_pile + n_bg:] = 90_000 + 20_000 - 1
    chrom = np.zeros(s.shape[0], dtype=np.int32)
    st = np.zeros(s.shape[0], dtype=np.int8)
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    o_mask, g_mask = both_regions([0, 0], [99_900, 250_000], [100_200, 251_000], [1, -1], 1)
    return o_reads, g_reads, o_mask, g_mask


@pytest.mark.parametrize("n_pile,narrow", [(65_535, True), (65_536, False)])
def test_bound_at_65535_reads(rb, n_pile, narrow):
    o_reads, g_reads, o_mask, g_mask = _pileup(rb, n_pile)
    cov = rb.calcCoverage(g_reads, g_mask)
    assert storage_bytes(rb, cov) == (2 if narrow else 4)
    got = cov.to_list()
    assert got[0].max() == n_pile
    assert_coverage_equal(got, O.calc_coverage(o_reads, o_mask))
    m = np.asarray(rb.binCoverageMatrix(cov, binSize=30))
    assert m[0].max() == n_pile                         # bins of 10 bases inside the pile-up


@pytest.mark.parametrize("n_pile,narrow", [(65_000, True), (65_001, False)])
def test_bound_counts_long_reads_through_the_binned_index(rb, n_pile, narrow):
    o_reads, g_reads, o_mask, g_mask = _pileup(rb, n_pile, n_long=535)
    rb.calcCoverage(g_reads, rb.GRangesList(g_mask, np.array([0, 1, 2], dtype=np.int64)))   # builds the index
    cov = rb.calcCoverage(g_reads, g_mask)
    assert storage_bytes(rb, cov) == (2 if narrow else 4)
    got = cov.to_list()
    assert got[0].max() == n_pile + 535
    assert_coverage_equal(got, O.calc_coverage(o_reads, o_mask))


def test_na_seqlength_rule_on_narrow_storage(rb):
    rng = np.random.default_rng(61)
    true_len = [30000, 8000]
    chrom, s, e, st = synth_reads(rng, 5000, true_len, width=(20, 90))
    keep = ~((chrom == 0) & (s > 20000))
    chrom, s, e, st = chrom[keep], s[keep], e[keep], st[keep]
    na_len = np.asarray([-1, 8000], dtype=np.int64)
    o_reads = O.Reads(chrom, s, e, st, na_len)
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=["c0", "c1"], seqlengths=na_len)
    rc = rng.integers(0, 2, size=300)
    rs = rng.integers(1, 7000, size=300)
    rs[rc == 0] = rng.integers(1, 25000, size=int((rc == 0).sum()))
    re_ = rs + rng.integers(0, 900, size=300)
    rst = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=300)
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 2)
    want = O.calc_coverage(o_reads, o_mask)
    cov = rb.calcCoverage(g_reads, g_mask)
    assert storage_bytes(rb, cov) == 2
    assert_coverage_equal(cov.to_list(), want)
    assert 0 < sum(w is None for w in want) < len(want)


def test_concat3_of_narrow_and_wide_handles(rb, monkeypatch):
    rng = np.random.default_rng(71)
    clen = [200_000]
    chrom, s, e, st = synth_reads(rng, 40_000, clen, width=(30, 80))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    rs = rng.integers(1000, 190_000, size=200)
    rst = rng.choice(np.array([1, -1], dtype=np.int8), size=200)
    parts = []
    for k, (a, b) in enumerate([(-500, -1), (0, 700), (701, 1200)]):
        if k == 1:                                      # the list-path centre of C4 is int32 too
            monkeypatch.setenv("RCP_COVERAGE_WIDE", "1")
        else:
            monkeypatch.delenv("RCP_COVERAGE_WIDE", raising=False)
        o_m, g_m = both_regions(np.zeros(200, int), rs + a, rs + b, rst, 1)
        cov = rb.calcCoverage(g_reads, g_m)
        assert storage_bytes(rb, cov) == (4 if k == 1 else 2)
        parts.append((cov, O.calc_coverage(o_reads, o_m)))
    from recoup_b200.coverage import _concat3
    cat = _concat3(parts[0][0], parts[1][0], parts[2][0], None)
    assert storage_bytes(rb, cat) == 4
    got = cat.to_list()
    for r in range(200):
        pieces = [p[1][r] for p in parts]
        if any(x is None for x in pieces):
            continue
        assert np.array_equal(got[r].astype(np.int64), np.concatenate(pieces))
