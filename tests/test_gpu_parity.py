"""Parity tests proper: the CUDA library, called through the C ABI (via the host mirror), against
the oracle on the same seeded inputs.  Coverage must be BIT-EXACT; profile matrices within
1e-6 relative (north_star).  Run with `-m gpu` on a B200."""
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import recoup_oracle as O
from tests.helpers import (assert_coverage_equal, assert_matrix_close, both_reads, both_regions,
                           fixture_exons, fixture_genes, fixture_reads, synth_reads)

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# C1: the reference's bundled fixture
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 1])
def test_c1_fixture_tss_100_bins(gpu, fixture_data, k):
    rb = gpu
    o_reads, g_reads = fixture_reads(fixture_data, k)
    o_genes, g_genes = fixture_genes(fixture_data)
    want_cov = O.coverage_ref(o_reads, o_genes, "tss", (2000, 2000))
    inp = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRef(inp, g_genes, "tss", (2000, 2000))
    cov = inp[0]["coverage"]
    assert cov.names == list(fixture_data["gene_names"])
    assert cov.n_null == (6 if k == 0 else 4)
    assert_coverage_equal(cov.to_list(), want_cov)
    bp = dict(flankBinSize=0, regionBinSize=100, sumStat="mean", interpolation="auto")
    rb.profileMatrix(inp, (2000, 2000), bp)
    m = inp[0]["profile"]
    assert m.shape == (100, 100) and m.flags.f_contiguous and m.rownames == cov.names
    assert_matrix_close(m, O.profile_matrix(want_cov, (2000, 2000), bp))


@pytest.mark.parametrize("region,flank,bp", [
    ("tes", (1000, 3000), dict(flankBinSize=0, regionBinSize=0)),
    ("tss", (500, 1500), dict(flankBinSize=0, regionBinSize=64, sumStat="median")),
    ("genebody", (2000, 2000), dict(flankBinSize=50, regionBinSize=150, sumStat="mean",
                                    interpolation="auto")),
    ("genebody", (2000, 1000), dict(flankBinSize=0, regionBinSize=60, sumStat="median",
                                    interpolation="spline")),
    ("genebody", (0, 1000), dict(flankBinSize=30, regionBinSize=200, sumStat="mean",
                                 interpolation="auto")),
])
def test_fixture_regions_and_profiles(gpu, fixture_data, region, flank, bp):
    rb = gpu
    o_reads, g_reads = fixture_reads(fixture_data, 0)
    o_genes, g_genes = fixture_genes(fixture_data)
    want_cov = O.coverage_ref(o_reads, o_genes, region, flank)
    inp = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRef(inp, g_genes, region, flank)
    assert_coverage_equal(inp[0]["coverage"].to_list(), want_cov)
    rb.profileMatrix(inp, flank, bp)
    assert_matrix_close(inp[0]["profile"], O.profile_matrix(want_cov, flank, bp))


def test_fixture_rna(gpu, fixture_data):
    rb = gpu
    o_reads, g_reads = fixture_reads(fixture_data, 0)
    o_genes, g_genes = fixture_genes(fixture_data)
    o_ex, g_ex = fixture_exons(fixture_data)
    want = O.coverage_rna_ref(o_reads, o_ex, o_genes, (2000, 2000))
    inp = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRnaRef(inp, g_ex, g_genes, (2000, 2000))
    cov = inp[0]["coverage"]
    assert cov.names == list(fixture_data["exon_gene_names"])
    assert_coverage_equal(cov.to_list(), want)
    bp = dict(flankBinSize=50, regionBinSize=150, sumStat="mean", interpolation="auto")
    rb.profileMatrix(inp, (2000, 2000), bp)
    assert_matrix_close(inp[0]["profile"], O.profile_matrix(want, (2000, 2000), bp))
    # the centre part alone is calcCoverage over the GRangesList
    center = rb.calcCoverage(g_reads, g_ex)
    assert_coverage_equal(center.to_list(), O.calc_coverage(o_reads, o_ex))


# ------------------------------------------------------------------------------------------------
# synthetic: every NULL / strand / size rule
# ------------------------------------------------------------------------------------------------
def _regions(rng, n, clen, lengths):
    clen = np.asarray(clen)
    chrom = rng.integers(0, clen.shape[0], size=n)
    L = rng.choice(np.asarray(lengths), size=n)
    start = (rng.random(n) * (clen[chrom] + 300)).astype(np.int64) - 150
    strand = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=n)
    return chrom, start, start + L - 1, strand


@pytest.mark.parametrize("seed", [11, 12])
@pytest.mark.parametrize("ignore,filt", [(True, None), (False, None), (True, "+"), (False, "-"),
                                         (True, "*")])
def test_random_regions_all_strand_modes(gpu, seed, ignore, filt):
    rb = gpu
    rng = np.random.default_rng(seed)
    clen = [30000, 70000, 900, 15000]
    chrom, s, e, st = synth_reads(rng, 20000, clen, width=(1, 400))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    # lengths straddling the warp kernel (<= 1024), one tile and many tiles
    rc, rs, re_, rst = _regions(rng, 300, clen, [1, 2, 31, 32, 33, 127, 128, 129, 1000, 1023,
                                                 1024, 1025, 4095, 4096, 4097, 8192, 9000, 20011])
    rs[:4] = [0, -1, 1, 2]
    re_[:4] = rs[:4] + [500, 500, 2000, 5000]
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    filt_code = None if filt is None else {"+": 1, "-": -1, "*": 0}[filt]
    want = O.calc_coverage(o_reads, o_mask, filt_code, ignore)
    got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
    assert_coverage_equal(got.to_list(), want)
    lens = got.lengths()
    assert [int(l) for l in lens] == [0 if w is None else len(w) for w in want]
    assert any(w is None for w in want) and sum(w is not None for w in want) > 50


def test_bucket_path_overlapping_regions_and_hit_list_overflow(gpu, monkeypatch):
    """Heavily overlapping regions give several hits per read (overflow runs of the cell table);
    a hit list that is too small makes pass 2 walk the reads again.  Same results either way."""
    rb = gpu
    rng = np.random.default_rng(31)
    clen = [120000, 40000]
    chrom, s, e, st = synth_reads(rng, 40000, clen, width=(1, 3000))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    # 40 copies of the same few windows + nested windows + random ones, all strands
    rc, rs, re_, rst = _regions(rng, 200, clen, [50, 500, 1024, 1025, 3000, 7168, 7169, 30000])
    rc = np.concatenate([rc, np.zeros(120, dtype=rc.dtype)])
    rs = np.concatenate([rs, np.tile([5000, 5000, 5100], 40)])
    re_ = np.concatenate([re_, np.tile([5999, 25999, 5300], 40)])
    rst = np.concatenate([rst, rng.choice(np.array([1, -1, 0], dtype=np.int8), size=120)])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    for ignore, filt in [(True, None), (False, None), (False, "+")]:
        filt_code = None if filt is None else {"+": 1, "-": -1, "*": 0}[filt]
        want = O.calc_coverage(o_reads, o_mask, filt_code, ignore)
        monkeypatch.delenv("RCP_BKT_HIT_CAP", raising=False)
        got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
        assert_coverage_equal(got.to_list(), want)
        monkeypatch.setenv("RCP_BKT_HIT_CAP", "100")
        got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
        assert_coverage_equal(got.to_list(), want)
        # dense mask + "very many" reads: the automatic path hands the call to the sorted index
        monkeypatch.setenv("RCP_BKT_SWITCH_READS", "1000")
        got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
        assert_coverage_equal(got.to_list(), want)
        monkeypatch.delenv("RCP_BKT_SWITCH_READS", raising=False)
        monkeypatch.delenv("RCP_BKT_HIT_CAP", raising=False)
    monkeypatch.delenv("RCP_BKT_HIT_CAP", raising=False)


def test_pileups_long_reads_and_no_strand(gpu):
    rb = gpu
    rng = np.random.default_rng(21)
    clen = [200000]
    # 5000 duplicates at one position (warp-aggregated atomics), very long reads (rank method is
    # width independent), plus background
    chrom, s, e, st = synth_reads(rng, 30000, clen, width=(30, 60))
    s[:5000] = 77777
    e[:5000] = 77777 + 49
    s[5000:5050] = rng.integers(1, 50000, size=50)
    e[5000:5050] = s[5000:5050] + rng.integers(60000, 120000, size=50)
    o_reads = O.Reads(chrom, s, e, np.zeros_like(st), clen)
    g_reads = rb.GRanges(chrom, s, e, seqlevels=["c0"], seqlengths=clen)          # no strand given
    rc, rs, re_, rst = _regions(rng, 200, clen, [200, 1000, 5000, 30000])
    rs[0], re_[0] = 77000, 79999
    rs[1], re_[1] = 1, 200000
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 1)
    want = O.calc_coverage(o_reads, o_mask)
    got = rb.calcCoverage(g_reads, g_mask)
    assert_coverage_equal(got.to_list(), want)
    assert want[0].max() >= 5000
    # ignore.strand=FALSE with strandless reads: '*' reads match every region
    got2 = rb.calcCoverage(g_reads, g_mask, ignore_strand=False)
    assert_coverage_equal(got2.to_list(), want)
    # a strand pre-filter sees only '*' reads: "+" keeps none (every region NULL), "*" keeps all
    for filt, code in (("+", 1), ("-", -1), ("*", 0)):
        want_f = O.calc_coverage(o_reads, o_mask, code, True)
        got_f = rb.calcCoverage(g_reads, g_mask, strand=filt)
        assert_coverage_equal(got_f.to_list(), want_f)
        assert all(w is None for w in want_f) == (filt != "*")


def test_groups_denser_than_shared_memory(gpu):
    """Split path: a 64-kb group holding more candidates than its CTA's shared memory (the group
    kernel scatters it directly), one of them with 70 000 reads in ONE 1-kb sub-bin."""
    rb = gpu
    rng = np.random.default_rng(33)
    clen = [400000]
    n_bg, n_pile = 170000, 70000
    chrom = np.zeros(n_bg + n_pile, dtype=np.int32)
    w = rng.integers(20, 90, size=n_bg + n_pile)
    s = np.empty(n_bg + n_pile, dtype=np.int64)
    s[:n_bg] = rng.integers(1, 130000, size=n_bg)                  # two groups, ~85 000 candidates each
    s[n_bg:] = rng.integers(262144 + 5 * 1024, 262144 + 6 * 1024 - 100, size=n_pile)   # one sub-bin
    e = s + w - 1
    st = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=n_bg + n_pile)
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    rc, rs, re_, rst = _regions(rng, 60, clen, [500, 3000, 20000])
    rs[0], re_[0] = 1, 135000
    rs[1], re_[1] = 262144, 262144 + 9000
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 1)
    for ignore in (True, False):
        want = O.calc_coverage(o_reads, o_mask, None, ignore)
        got = rb.calcCoverage(g_reads, g_mask, ignore_strand=ignore)
        assert_coverage_equal(got.to_list(), want)
    # the same reads through the handle's binned index (GRangesList mask)
    ptr = np.arange(0, 61, 3, dtype=np.int64)
    o_list = dict(ptr=ptr, **o_mask)
    grl = rb.GRangesList(g_mask, ptr)
    want = O.calc_coverage(o_reads, o_list)
    got = rb.calcCoverage(g_reads, grl)
    assert_coverage_equal(got.to_list(), want)


@pytest.mark.parametrize("frag_len", [0, 150])
@pytest.mark.parametrize("ignore", [True, False])
def test_unknown_seqlengths_end_the_coverage_vector_at_the_last_overlapping_read(gpu, frag_len, ignore):
    """coverage.R:201 with NA seqlengths: coverage(reads)[[chr]] is as long as the largest end among the
    reads that overlap the region, so a window is NULL unless a read reaches its last position."""
    rb = gpu
    rng = np.random.default_rng(61)
    true_len = [30000, 8000, 500]
    chrom, s, e, st = synth_reads(rng, 5000, true_len, width=(20, 90))
    keep = ~((chrom == 0) & (s > 20000))               # nothing on the last third of c0
    chrom, s, e, st = chrom[keep], s[keep], e[keep], st[keep]
    na_len = np.asarray([-1, 8000, -1], dtype=np.int64)           # c0 and c2 unknown, c1 known
    es, ee = O.extend_fragments(s, e, st, frag_len, chrom, np.asarray([10**9, 8000, 10**9])) if frag_len else (s, e)
    o_reads = O.Reads(chrom, es, ee, st, na_len)
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=["c0", "c1", "c2"], seqlengths=na_len)
    rc, rs, re_, rst = _regions(rng, 300, true_len, [1, 30, 200, 1024, 1500, 6000])
    rc[:4], rs[:4], re_[:4], rst[:4] = [0, 0, 2, 1], [1, 19000, 1, 1], [30000, 23000, 500, 8000], [1, -1, 0, 1]
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 3)
    want = O.calc_coverage(o_reads, o_mask, None, ignore)
    got = rb.calcCoverage(g_reads, g_mask, ignore_strand=ignore, frag_len=frag_len)
    assert_coverage_equal(got.to_list(), want)
    n_null = sum(w is None for w in want)
    assert 0 < n_null < len(want) and got.n_null == n_null
    # the same windows with the lengths known: fewer NULLs (the rule is what makes the difference)
    o_known = O.Reads(chrom, es, ee, st, np.asarray([40000, 8000, 600]))
    assert sum(w is None for w in O.calc_coverage(o_known, o_mask, None, ignore)) < n_null
    # GRangesList masks: the largest range end of the element decides
    ptr = np.concatenate((np.arange(0, 300, 4), [300])).astype(np.int64)
    for g in range(ptr.shape[0] - 1):                   # one chromosome and strand per element
        rc[ptr[g]:ptr[g + 1]] = rc[ptr[g]]
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 3)
    want = O.calc_coverage(o_reads, dict(ptr=ptr, **o_mask), None, ignore)
    got = rb.calcCoverage(g_reads, rb.GRangesList(g_mask, ptr), ignore_strand=ignore, frag_len=frag_len)
    assert_coverage_equal(got.to_list(), want)
    assert any(w is None for w in want) and any(w is not None for w in want)
    # profile matrix of the NA coverage: NULL rows are zero rows (profile.R:6-12)
    o_mask1, g_mask1 = both_regions(rc[:100], rs[:100], rs[:100] + 399, rst[:100], 3)
    want = O.calc_coverage(o_reads, o_mask1, None, ignore)
    cov = rb.calcCoverage(g_reads, g_mask1, ignore_strand=ignore, frag_len=frag_len)
    assert_coverage_equal(cov.to_list(), want)
    inp = [dict(id="s", name="s", coverage=cov)]
    bp = dict(flankBinSize=0, regionBinSize=20, sumStat="mean", interpolation="auto")
    rb.profileMatrix(inp, (200, 200), bp)
    want_m = O.profile_matrix(want, (200, 200), bp)
    assert_matrix_close(inp[0]["profile"], want_m)
    # rcp_coverage_profile composes the two stages for such reads (the rule needs the coverage)
    m, is_null = rb.coverageProfile(g_reads, g_mask1, 20, ignore_strand=ignore, frag_len=frag_len)
    assert_matrix_close(m, want_m)
    assert np.array_equal(is_null, np.asarray([w is None for w in want]))


def test_empty_inputs(gpu):
    rb = gpu
    clen = [1000]
    none = rb.GRanges(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32),
                      seqlevels=["c0"], seqlengths=clen)
    _, g_mask = both_regions([0, 0], [1, 10], [100, 20], [1, -1], 1)
    cov = rb.calcCoverage(none, g_mask)
    assert cov.to_list() == [None, None] and cov.n_null == 2                  # no reads: all NULL
    m = rb.binCoverageMatrix(cov, binSize=5)
    assert m.shape == (2, 5) and (np.asarray(m) == 0).all()
    some = rb.GRanges(np.zeros(2, np.int32), [5, 50], [30, 80], seqlevels=["c0"], seqlengths=clen)
    empty_mask = rb.GRanges(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32),
                            seqlevels=["c0"])
    cov0 = rb.calcCoverage(some, empty_mask)
    assert len(cov0) == 0 and cov0.to_list() == []
    # a region on a chromosome the reads do not know -> NULL (coverage.R:194-197)
    other = rb.GRanges(["cX", "c0"], [5, 5], [30, 30], strand=["+", "+"], seqlevels=["cX", "c0"])
    cov1 = rb.calcCoverage(some, other)
    got = cov1.to_list()
    assert got[0] is None and got[1].tolist() == [1] * 26


def test_fragment_extension(gpu):
    rb = gpu
    rng = np.random.default_rng(31)
    clen = [40000, 9000]
    chrom, s, e, st = synth_reads(rng, 8000, clen, width=(36, 36))
    s[:10] = 1
    e[:10] = 36
    es, ee = O.extend_fragments(s, e, st, 200, chrom, clen)
    o_reads = O.Reads(chrom, es, ee, st, clen)
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=["c0", "c1"], seqlengths=clen)
    rc, rs, re_, rst = _regions(rng, 60, clen, [500, 3000])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 2)
    want = O.calc_coverage(o_reads, o_mask)
    got = rb.calcCoverage(g_reads, g_mask, frag_len=200)
    assert_coverage_equal(got.to_list(), want)


@pytest.mark.parametrize("ignore,filt", [(False, None), (True, "+"), (False, "-"), (True, None)])
def test_uniform_width_index_with_trimmed_exceptions(gpu, ignore, filt):
    """Fixed-width libraries use the one-sort index (ends = starts + w); reads trimmed at a
    chromosome end are the exceptions carried by the correction source.  All strand modes."""
    rb = gpu
    rng = np.random.default_rng(33)
    clen = [6000, 2500, 400]
    chrom, s, e, st = synth_reads(rng, 12000, clen, width=(36, 36))
    s[:40] = rng.integers(1, 30, size=40)                # pile reads onto the chromosome starts
    e[:40] = s[:40] + 35
    es, ee = O.extend_fragments(s, e, st, 200, chrom, clen)
    assert 0 < int(((ee - es + 1) != 200).sum()) < 4096   # some, but few, exceptions
    o_reads = O.Reads(chrom, es, ee, st, clen)
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=["c0", "c1", "c2"], seqlengths=clen)
    rc, rs, re_, rst = _regions(rng, 150, clen, [1, 50, 199, 200, 201, 399, 1024, 1500, 2400])
    rs[:6] = [1, 1, 1, 5800, 2300, 1]
    re_[:6] = [100, 250, 6000, 6000, 2500, 400]
    rc[:6] = [0, 1, 0, 0, 1, 2]
    o_mask, g_mask = both_regions(rc, rs, re_, rst, 3)
    filt_code = None if filt is None else {"+": 1, "-": -1, "*": 0}[filt]
    want = O.calc_coverage(o_reads, o_mask, filt_code, ignore)
    got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore, frag_len=200)
    assert_coverage_equal(got.to_list(), want)


@pytest.mark.parametrize("ignore,filt", [(False, None), (True, "-")])
def test_uniform_width_fixture_stranded(gpu, fixture_data, ignore, filt):
    rb = gpu
    o_reads, g_reads = fixture_reads(fixture_data, 1)          # every read is 180 bp wide
    o_genes, g_genes = fixture_genes(fixture_data)
    filt_code = None if filt is None else {"+": 1, "-": -1}[filt]
    want = O.coverage_ref(o_reads, o_genes, "genebody", (1500, 500), filt_code, ignore)
    inp = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRef(inp, g_genes, "genebody", (1500, 500),
                   strandedParams=dict(strand=filt, ignoreStrand=ignore))
    assert_coverage_equal(inp[0]["coverage"].to_list(), want)


@pytest.mark.parametrize("ignore", [True, False])
def test_granges_list_multiplicity(gpu, ignore):
    rb = gpu
    rng = np.random.default_rng(41)
    clen = [60000, 25000]
    chrom, s, e, st = synth_reads(rng, 15000, clen, width=(20, 1500))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    ptr, xc, xs, xe, xst = [0], [], [], [], []
    for g in range(80):
        c = int(rng.integers(0, 2))
        ne = int(rng.integers(1, 12))
        pos = int(rng.integers(1, clen[c] - 12000))
        gst = int(rng.choice([1, -1, 0]))
        ex = []
        for _ in range(ne):
            w = int(rng.integers(1, 700))
            ex.append((pos, pos + w - 1))
            pos += w + int(rng.integers(1, 400))
        if g % 7 == 0:
            ex = ex[::-1]                       # list order is respected, not genomic order
        if g % 11 == 0 and ne > 1:
            ex[1] = (ex[0][0] + 3, ex[0][1] + 9)    # overlapping ranges
        for a, b in ex:
            xc.append(c); xs.append(a); xe.append(b); xst.append(gst)
        ptr.append(len(xs))
    ptr.append(len(xs))                         # empty element -> NULL
    # one giant element (> 4096 stitched bases -> several tiles)
    for q in range(30):
        xc.append(0); xs.append(2000 + q * 900); xe.append(2000 + q * 900 + 499); xst.append(-1)
    ptr.append(len(xs))
    o_mask = dict(ptr=ptr, chrom=xc, start=xs, end=xe, strand=xst)
    u = rb.GRanges(np.asarray(xc, np.int32), xs, xe, strand=np.asarray(xst, np.int8),
                   seqlevels=["c0", "c1"])
    g_mask = rb.GRangesList(u, ptr)
    want = O.calc_coverage(o_reads, o_mask, None, ignore)
    got = rb.calcCoverage(g_reads, g_mask, ignore_strand=ignore)
    assert_coverage_equal(got.to_list(), want)
    assert want[-2] is None and want[-1] is not None and len(want[-1]) == 15000


# ------------------------------------------------------------------------------------------------
# profile matrix
# ------------------------------------------------------------------------------------------------
def _gene_like_coverage(rb, rng, n_regions=120, flank=(300, 200)):
    clen = [400000]
    chrom, s, e, st = synth_reads(rng, 60000, clen, width=(50, 150))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    w = rng.choice([1, 3, 9, 40, 55, 70, 100, 500, 3000, 9000], size=n_regions)
    gs = rng.integers(1000, 380000, size=n_regions)
    gst = rng.choice(np.array([1, -1], dtype=np.int8), size=n_regions)
    s2, e2 = O.get_regional_ranges(gs, gs + w - 1, gst, "genebody", flank)
    o_mask, g_mask = both_regions(np.zeros(n_regions, int), s2, e2, gst, 1)
    want = O.calc_coverage(o_reads, o_mask)
    got = rb.calcCoverage(g_reads, g_mask)
    return want, got


@pytest.mark.parametrize("bp", [
    dict(flankBinSize=20, regionBinSize=60, sumStat="mean", interpolation="auto"),
    dict(flankBinSize=20, regionBinSize=60, sumStat="median", interpolation="auto"),
    dict(flankBinSize=0, regionBinSize=45, sumStat="mean", interpolation="spline"),
    dict(flankBinSize=7, regionBinSize=50, sumStat="median", interpolation="spline"),
    dict(flankBinSize=33, regionBinSize=257, sumStat="mean", interpolation="auto"),
])
def test_unequal_length_profiles(gpu, bp):
    rb = gpu
    rng = np.random.default_rng(51)
    flank = (300, 200)
    want_cov, got_cov = _gene_like_coverage(rb, rng, flank=flank)
    assert_coverage_equal(got_cov.to_list(), want_cov)
    want = O.profile_matrix(want_cov, flank, bp)
    inp = [dict(id="s", name="s", coverage=got_cov)]
    rb.profileMatrix(inp, flank, bp)
    assert_matrix_close(inp[0]["profile"], want)


@pytest.mark.parametrize("interp", ["auto", "spline", "neighborhood"])
@pytest.mark.parametrize("stat", ["mean", "median"])
def test_interpolation_kernels(gpu, interp, stat):
    """Segments shorter than the bin count (util.R:17-73): spline, neighbourhood and the 'auto'
    switch at (n - L) / n < 0.2."""
    rb = gpu
    rng = np.random.default_rng(61)
    clen = [50000]
    chrom, s, e, st = synth_reads(rng, 30000, clen, width=(20, 90))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    n_bins = 40
    lengths = np.array([4, 5, 7, 12, 20, 31, 32, 33, 35, 38, 39, 40, 41, 80, 200])
    if interp != "neighborhood":
        lengths = np.concatenate([[1, 2, 3], lengths])
    starts = rng.integers(100, 45000, size=lengths.shape[0])
    strand = rng.choice(np.array([1, -1], dtype=np.int8), size=lengths.shape[0])
    o_mask, g_mask = both_regions(np.zeros(len(lengths), int), starts, starts + lengths - 1, strand, 1)
    want_cov = O.calc_coverage(o_reads, o_mask)
    got_cov = rb.calcCoverage(g_reads, g_mask)
    assert_coverage_equal(got_cov.to_list(), want_cov)
    want = O.bin_coverage_matrix(want_cov, n_bins, stat, interp)
    got = rb.binCoverageMatrix(got_cov, binSize=n_bins, stat=stat, interpolation=interp)
    assert_matrix_close(got, want)
    assert got.colnames == [str(i + 1) for i in range(n_bins)]


def test_rounding_sample_kind_and_scale(gpu):
    rb = gpu
    rng = np.random.default_rng(71)
    want_cov, got_cov = _gene_like_coverage(rb, rng, n_regions=40)
    bp = dict(flankBinSize=20, regionBinSize=60, sumStat="mean", interpolation="auto")
    want = O.profile_matrix(want_cov, (300, 200), bp, sample_kind="Rounding")
    inp = [dict(id="s", name="s", coverage=got_cov)]
    rb.profileMatrix(inp, (300, 200), bp, sample_kind="Rounding")
    assert_matrix_close(inp[0]["profile"], want)
    # linear normalisation (recoup.R:559-577): coverage * factor before binning
    got_cov.set_scale(0.37)
    inp = [dict(id="s", name="s", coverage=got_cov)]
    rb.profileMatrix(inp, (300, 200), bp)
    want_scaled = O.profile_matrix([None if c is None else c * 0.37 for c in want_cov],
                                   (300, 200), bp)
    assert_matrix_close(inp[0]["profile"], want_scaled)


def test_per_base_matrix_and_linear_interp_error(gpu):
    rb = gpu
    rng = np.random.default_rng(81)
    clen = [90000]
    chrom, s, e, st = synth_reads(rng, 20000, clen, width=(30, 70))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    sites = rng.integers(600, 89000, size=333)
    sst = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=333)
    s2, e2 = O.get_regional_ranges(sites, sites, sst, "custom", (500, 500))
    o_mask, g_mask = both_regions(np.zeros(333, int), s2, e2, sst, 1)
    want_cov = O.calc_coverage(o_reads, o_mask)
    got_cov = rb.calcCoverage(g_reads, g_mask)
    assert_coverage_equal(got_cov.to_list(), want_cov)
    bp = dict(flankBinSize=0, regionBinSize=0)
    inp = [dict(id="s", name="s", coverage=got_cov)]
    rb.profileMatrix(inp, (500, 500), bp)
    want = O.profile_matrix(want_cov, (500, 500), bp)
    assert inp[0]["profile"].shape == (333, 1000)
    assert np.array_equal(np.asarray(inp[0]["profile"]), want)          # integers: exact
    up = rb.baseCoverageMatrix(got_cov, flank=(37, 90), where="upstream")
    dn = rb.baseCoverageMatrix(got_cov, flank=(37, 90), where="downstream")
    assert np.array_equal(np.asarray(up), O.base_coverage_matrix(want_cov, (37, 90), "upstream"))
    assert np.array_equal(np.asarray(dn), O.base_coverage_matrix(want_cov, (37, 90), "downstream"))
    with pytest.raises(rb.RecoupError) as ei:
        rb.binCoverageMatrix(got_cov, binSize=10, interpolation="linear")
    assert ei.value.code == 5 and "inear" in str(ei.value)


# ------------------------------------------------------------------------------------------------
# size-independent properties at a larger size + the C twin as a mid-size checker
# ------------------------------------------------------------------------------------------------
def test_midsize_against_c_oracle_and_properties(gpu):
    rb = gpu
    rng = np.random.default_rng(91)
    clen = [3_000_000, 1_500_000, 700_000]
    n = 1_500_000
    chrom, s, e, st = synth_reads(rng, n, clen, width=(200, 200))
    g_reads = rb.GRanges(chrom, s, e, strand=st, seqlevels=["a", "b", "c"], seqlengths=clen)
    R = 3000
    tss = rng.integers(6000, 600_000, size=R)
    rc = rng.integers(0, 3, size=R)
    rst = rng.choice(np.array([1, -1], dtype=np.int8), size=R)
    s2, e2 = O.get_regional_ranges(tss, tss, rst, "tss", (5000, 5000))
    g_mask = rb.GRanges(rc.astype(np.int32), s2, e2, strand=rst, seqlevels=["a", "b", "c"])
    cov = rb.calcCoverage(g_reads, g_mask)
    ix = CO.Index(chrom, s, e, st, clen)
    dense = CO.coverage(ix, rc, s2, e2, rst)
    assert_coverage_equal(cov.to_list(), dense.to_list())
    bp = dict(flankBinSize=0, regionBinSize=200)
    inp = [dict(id="s", name="s", coverage=cov)]
    rb.profileMatrix(inp, (5000, 5000), bp)
    m = np.asarray(inp[0]["profile"])
    assert_matrix_close(m, CO.profile_matrix(dense, (5000, 5000), bp, True))
    # property: a row's mean * 10000 == bases of reads inside the window (checksum of checksums)
    got_rows = m.mean(axis=1) * 10000
    lens = dense.len
    for r in rng.integers(0, R, size=50):
        if lens[r] == 0:
            continue
        on = chrom == rc[r]
        ov = np.minimum(e[on], e2[r]) - np.maximum(s[on], s2[r]) + 1
        assert abs(got_rows[r] - ov[ov > 0].sum()) < 1e-6 * max(1.0, got_rows[r])
    # linearity: coverage(A u B) == coverage(A) + coverage(B) wherever all three are non-NULL
    half = n // 2
    ga = rb.GRanges(chrom[:half], s[:half], e[:half], strand=st[:half], seqlevels=["a", "b", "c"],
                    seqlengths=clen)
    gb = rb.GRanges(chrom[half:], s[half:], e[half:], strand=st[half:], seqlevels=["a", "b", "c"],
                    seqlengths=clen)
    sub = rb.GRanges(rc[:200].astype(np.int32), s2[:200], e2[:200], strand=rst[:200],
                     seqlevels=["a", "b", "c"])
    ca = rb.calcCoverage(ga, sub).to_list()
    cb = rb.calcCoverage(gb, sub).to_list()
    call = cov.fetch(0, 200)
    for x, y, zed in zip(ca, cb, call):
        if zed is None:
            assert x is None and y is None
        else:
            xx = np.zeros_like(zed) if x is None else x
            yy = np.zeros_like(zed) if y is None else y
            assert np.array_equal(xx + yy, zed)
    # strand symmetry: flipping the region strand reverses the vector
    flipped = rb.GRanges(rc[:200].astype(np.int32), s2[:200], e2[:200], strand=-rst[:200],
                         seqlevels=["a", "b", "c"])
    cf = rb.calcCoverage(g_reads, flipped).to_list()
    for x, y in zip(cf, call):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x[::-1], y)


def test_handles_and_errors(gpu):
    rb = gpu
    from recoup_b200 import _lib
    assert _lib.lib.rcp_coverage_free(987654) == _lib.RCP_ERR_HANDLE
    assert _lib.lib.rcp_reads_free(987654) == _lib.RCP_ERR_HANDLE
    bad = rb.GRanges(np.zeros(2, np.int32), [5, 0], [30, 9], seqlevels=["c0"], seqlengths=[100])
    mask = rb.GRanges(np.zeros(1, np.int32), [1], [10], seqlevels=["c0"])
    with pytest.raises(rb.RecoupError) as ei:
        rb.calcCoverage(bad, mask)                      # a read with start < 1
    assert ei.value.code == _lib.RCP_ERR_DATA
    sm = C.c_int(0)
    assert _lib.lib.rcp_device_info(None, C.byref(sm), None, None, None) == 0 and sm.value >= 100
    before = _lib.lib.rcp_launch_count(1)
    ok = rb.GRanges(np.zeros(2, np.int32), [5, 20], [30, 90], seqlevels=["c0"], seqlengths=[100])
    cov = rb.calcCoverage(ok, mask)
    assert cov[0].tolist() == [0, 0, 0, 0, 1, 1, 1, 1, 1, 1]
    assert _lib.lib.rcp_launch_count(0) > 0 and before >= 0


@pytest.mark.parametrize("n_reads,runs", [(20000, "sorted"), (1, "sorted"), (4099, "many"),
                                          (5000, "empty_runs")])
def test_seqnames_as_runs_give_the_same_coverage(gpu, n_reads, runs):
    """rcp_reads_load_rle (seqnames as the Rle a GRanges holds) == the dense upload == oracle"""
    rb = gpu
    rng = np.random.default_rng(5)
    clen = [30000, 70000, 900, 15000]
    chrom, s, e, st = synth_reads(rng, n_reads, clen, width=(1, 300))
    if runs != "many":                       # grouped by chromosome, like a sorted BAM
        order = np.argsort(chrom, kind="stable")
        chrom, s, e, st = chrom[order], s[order], e[order], st[order]
    rle = rb.Rle.encode(chrom)
    if runs == "empty_runs":                 # zero-length runs between and around the real ones
        vals = np.repeat(rle.values, 3)
        lens = np.zeros(vals.shape[0], dtype=np.int32)
        lens[1::3] = rle.lengths
        vals[0::3] = 3 - vals[0::3]
        rle = rb.Rle(vals, lens)
    o_reads, g_dense = both_reads(chrom, s, e, st, clen)
    g_rle = rb.GRanges(rle, s, e, strand=st, seqlevels=g_dense.seqlevels, seqlengths=clen)
    assert np.array_equal(g_rle.seqnames, chrom)
    rc, rs, re_, rst = _regions(rng, 120, clen, [1, 33, 128, 1024, 1025, 5000, 9000])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    want = O.calc_coverage(o_reads, o_mask, None, False)
    # force the runs entry (the wrapper picks it by itself only when it pays)
    from recoup_b200.coverage import DeviceReads
    dr = DeviceReads(g_rle, 0, use_runs=True)
    g_rle._device[0] = dr
    got = rb.calcCoverage(g_rle, g_mask, ignore_strand=False)
    assert_coverage_equal(got.to_list(), want)
    assert_coverage_equal(rb.calcCoverage(g_dense, g_mask, ignore_strand=False).to_list(), want)
    dr.free()
    g_rle._device.clear()
    if runs == "sorted" and n_reads > 1:     # and through the wrapper, which now takes the runs
        assert g_rle.seqnames_rle.nrun * 2 < len(g_rle)
        assert_coverage_equal(rb.calcCoverage(g_rle, g_mask, ignore_strand=False).to_list(), want)


@pytest.mark.parametrize("frag_len", [0, 200])
@pytest.mark.parametrize("runs", [False, True])
def test_one_width_reads_upload_start_only(gpu, runs, frag_len):
    """rcp_reads_load_width (start + ONE width; the ends never cross PCIe) == the dense upload ==
    oracle, with and without the fragment extension, seqnames dense or as runs"""
    rb = gpu
    rng = np.random.default_rng(11)
    clen = [30000, 70000, 900, 15000]
    n, w = 6001, 36
    chrom, s, _, st = synth_reads(rng, n, clen, width=(w, w))
    s = np.minimum(s, np.asarray(clen)[chrom] - w + 1).astype(np.int32)
    if runs:
        order = np.argsort(chrom, kind="stable")
        chrom, s, st = chrom[order], s[order], st[order]
    e = (s + w - 1).astype(np.int32)
    o_reads, g_dense = both_reads(chrom, s, e, st, clen)
    g_w = rb.GRanges(rb.Rle.encode(chrom) if runs else chrom, s, width=w, strand=st,
                     seqlevels=g_dense.seqlevels, seqlengths=clen)
    rc, rs, re_, rst = _regions(rng, 150, clen, [1, 33, 128, 1024, 1025, 5000, 9000])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    got = rb.calcCoverage(g_w, g_mask, ignore_strand=False, frag_len=frag_len)
    assert g_w._end is None                     # the host never built the ends
    ref = rb.calcCoverage(g_dense, g_mask, ignore_strand=False, frag_len=frag_len)
    assert_coverage_equal(got.to_list(), ref.to_list())
    if frag_len:
        es, ee = O.extend_fragments(s, e, st, frag_len, chrom, clen)
        o_reads = O.Reads(chrom, es, ee, st, clen)
    assert_coverage_equal(got.to_list(), O.calc_coverage(o_reads, o_mask, None, False))
    # argument errors
    from recoup_b200 import _lib
    h = C.c_int(0)
    cl = np.asarray(clen, dtype=np.int64)
    rc_ = _lib.lib.rcp_reads_load_width(n, chrom.ctypes.data_as(C.c_void_p), 0, None, None,
                                        s.ctypes.data_as(C.c_void_p), 0, None, len(clen),
                                        cl.ctypes.data_as(C.POINTER(C.c_int64)), 0, _lib.MEM_HOST, C.byref(h))
    assert rc_ == _lib.RCP_ERR_ARG


def test_seqnames_runs_errors(gpu):
    rb = gpu
    from recoup_b200 import _lib
    s = np.arange(1, 9, dtype=np.int32)
    e = s + 5
    cl = np.asarray([100, 100], dtype=np.int64)

    def load(vals, lens):
        h = C.c_int(0)
        rv = np.asarray(vals, dtype=np.int32)
        rl = np.asarray(lens, dtype=np.int32)
        rc = _lib.lib.rcp_reads_load_rle(8, rv.shape[0], rv.ctypes.data_as(C.c_void_p),
                                         rl.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p),
                                         e.ctypes.data_as(C.c_void_p), None, 2,
                                         cl.ctypes.data_as(C.POINTER(C.c_int64)), 0, _lib.MEM_HOST,
                                         C.byref(h))
        if rc == 0:
            _lib.lib.rcp_reads_free(h.value)
        return rc

    assert load([0, 1], [5, 3]) == 0
    assert load([0, 1], [5, 2]) == _lib.RCP_ERR_DATA        # runs shorter than the reads
    assert load([0, 1], [5, 4]) == _lib.RCP_ERR_DATA        # ... longer
    assert load([0, 1], [9, -1]) == _lib.RCP_ERR_DATA       # negative run
    assert load([0, 2], [5, 3]) == _lib.RCP_ERR_DATA        # chromosome id out of range
    assert load([], []) == _lib.RCP_ERR_ARG


# ------------------------------------------------------------------------------------------------
# read import after the decode (SURVEY 8f N3)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("normalize", ["none", "downsample", "sampleto"])
@pytest.mark.parametrize("splice", ["keep", "remove"])
def test_preprocess_ranges_selection_on_the_device(gpu_auto, normalize, splice):
    rb = gpu_auto
    rng = np.random.default_rng(21)
    clen = [40000, 9000]
    libs = []
    for n in (6000, 4500, 5200):
        chrom, s, e, st = synth_reads(rng, n, clen, width=(20, 60))
        long_ = rng.random(n) < 0.2                       # "spliced" reads: much wider
        e = np.where(long_, np.minimum(e + rng.integers(200, 3000, size=n), np.asarray(clen)[chrom]), e)
        libs.append((chrom, s, e.astype(s.dtype), st))
    pp = {"normalize": normalize, "spliceAction": splice, "spliceRemoveQ": 0.75, "seed": 11,
          "sampleTo": 3000}
    inp = [{"name": "s%d" % i, "file": "s%d.bam" % i} for i in range(3)]

    def reader(x):
        c, s, e, st = libs[int(x["name"][1:])]
        return rb.GRanges(c, s, e, strand=st, seqlevels=["c0", "c1"], seqlengths=clen)

    rb.preprocessRanges(inp, pp, reader=reader)
    # oracle: the same steps on numpy arrays
    kept = []
    for c, s, e, st in libs:
        keep = O.splice_remove(s, e, 0.75)[0] if splice == "remove" else np.ones(len(s), bool)
        kept.append([a[keep] for a in (c, s, e, st)])
    idx = O.downsample_indices([len(k[0]) for k in kept], normalize, seed=11, sample_to=3000)
    rc, rs, re_, rst = _regions(rng, 60, clen, [1, 100, 1024, 1025, 5000])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    for x, k, ix in zip(inp, kept, idx):
        sel = k if ix is None else [a[ix - 1] for a in k]
        assert len(x["ranges"]) == len(sel[0])
        o_reads = O.Reads(sel[0], sel[1], sel[2], sel[3], np.asarray(clen))
        want = O.calc_coverage(o_reads, o_mask, None, False)
        got = rb.calcCoverage(x["ranges"], g_mask, ignore_strand=False)
        assert_coverage_equal(got.to_list(), want)
        if normalize != "none" or splice == "remove":
            assert np.array_equal(x["ranges"].start, sel[1]) and np.array_equal(x["ranges"].end, sel[2])
    if normalize == "downsample":
        assert len({len(x["ranges"]) for x in inp}) == 1


def test_width_quantile_and_selection_errors(gpu_auto):
    rb = gpu_auto
    from recoup_b200 import _lib
    rng = np.random.default_rng(22)
    s = rng.integers(1, 1000, size=5001).astype(np.int32)
    e = (s + rng.integers(0, 300, size=5001)).astype(np.int32)
    gr = rb.GRanges(np.zeros(5001, np.int32), s, e, seqlevels=["c"], seqlengths=[2000])
    for q in (0.0, 0.5, 0.75, 0.999, 1.0):
        keep, qu = O.splice_remove(s, e, q)
        got_q, got_n = rb.widthQuantile(gr, q)
        assert got_q == qu and got_n == int(keep.sum())
    bad = rb.SelectedGRanges(gr, 5001, idx=[1, 5002])
    with pytest.raises(rb.RecoupError) as ei:
        rb.device_reads(bad)
    assert ei.value.code == _lib.RCP_ERR_DATA
    none_left = rb.SelectedGRanges(gr, 0, max_width=0.5)
    mask = rb.GRanges(np.zeros(1, np.int32), [1], [50], seqlevels=["c"])
    assert rb.calcCoverage(none_left, mask)[0] is None          # no reads: NULL


# ------------------------------------------------------------------------------------------------
# consumers of the matrix (SURVEY 8f N4)
# ------------------------------------------------------------------------------------------------
def _consumer_matrices():
    rng = np.random.default_rng(77)
    a = rng.gamma(0.6, 3.0, size=(2001, 37))
    a[rng.random(a.shape) < 0.3] = 0.0                    # many ties at zero
    a[5] = 0.0
    b = np.round(rng.normal(0.0, 2.0, size=(64, 5)), 1)   # negatives, ties, even row count
    b[3, 2] = -0.0
    return [a, b, rng.random((1, 4)), rng.random((7, 1))]


@pytest.mark.parametrize("avgfun", ["mean", "median"])
@pytest.mark.parametrize("scale", ["natural", "log2"])
def test_plot_profiles_match_the_oracle(gpu_auto, avgfun, scale):
    rb = gpu_auto
    mats = [m for m in _consumer_matrices() if scale == "natural" or m.min() >= 0]
    opts = {"plotParams": {"sumStat": avgfun, "signalScale": scale, "smooth": False}}
    got = rb.calcPlotProfiles([{"profile": m} for m in mats], opts)
    for m, g in zip(mats, got):
        want = O.plot_profile(m, avgfun, scale)
        for k in ("profile", "upper", "lower"):
            assert np.allclose(g[k], want[k], rtol=1e-12, atol=1e-12, equal_nan=True), (k, m.shape)
    with pytest.raises(NotImplementedError):
        rb.calcPlotProfiles([{"profile": mats[0]}], {"plotParams": {"smooth": True}})


@pytest.mark.parametrize("what", ["sum1", "max2", "avg1", "suma", "maxa", "avga", "none"])
@pytest.mark.parametrize("order", ["descending", "ascending"])
def test_order_profiles_match_the_oracle(gpu_auto, what, order):
    rb = gpu_auto
    rng = np.random.default_rng(78)
    a = _consumer_matrices()[0]
    b = a[rng.permutation(a.shape[0])] * 1.5
    inp = [{"profile": a}, {"profile": b}]
    got = rb.orderProfiles(inp, {"orderBy": {"what": what, "order": order}})
    if what == "none":
        assert got["ix"].tolist() == list(range(1, a.shape[0] + 1))
        return
    kind, ref = what[:3], what[-1]
    if ref == "a":
        per = np.stack([O.row_order_values(x["profile"], kind) for x in inp], axis=1)
        val = O.row_order_values(per, kind)
    else:
        val = O.row_order_values(inp[int(ref) - 1]["profile"], kind)
    want = O.r_sort_index(val, order == "descending")
    # the ordering values agree to rounding; exact ties (zero rows) must come out in input order
    assert np.allclose(rb.rowStat(inp[0]["profile"], kind), O.row_order_values(a, kind), rtol=1e-13)
    gv = val[got["ix"] - 1]
    assert np.allclose(gv, val[want - 1], rtol=1e-12)
    zero = np.flatnonzero(val == 0) + 1
    assert [i for i in got["ix"] if val[i - 1] == 0] == zero.tolist()
    assert sorted(got["ix"].tolist()) == list(range(1, a.shape[0] + 1))


def test_sort_index_ties_nan_and_custom_order(gpu_auto):
    rb = gpu_auto
    v = np.array([3, 1, 2, 1, np.nan, 3.0, -0.0, 0.0, -np.inf, np.inf])
    for dec in (False, True):
        got = rb.sortIndex(v, dec)
        assert got["ix"].tolist() == O.r_sort_index(v, dec).tolist()
        assert np.array_equal(got["x"], v[got["ix"] - 1])
    got = rb.orderProfiles([], {"orderBy": {"custom": [5.0, 7.0, 5.0], "order": "descending"}})
    assert got["ix"].tolist() == [2, 1, 3]
    assert rb.sortIndex(np.zeros(0))["ix"].shape == (0,)
    rng = np.random.default_rng(3)
    big = np.round(rng.normal(size=300001), 2)
    assert np.array_equal(rb.sortIndex(big, True)["ix"], O.r_sort_index(big, True))


def test_matrix_quantile_and_heatmap_scale(gpu_auto):
    rb = gpu_auto
    from recoup_b200 import _lib
    mats = _consumer_matrices()
    probs = [0.0, 0.1, 0.5, 0.95, 0.96, 0.999, 1.0]
    for m in mats:
        assert np.allclose(rb.matrixQuantile(m, probs), O.r_quantile7(m, probs), rtol=1e-14, atol=0)
    inp = [{"profile": mats[0]}, {"profile": mats[0] * 2.0}]
    q95 = float(O.r_quantile7(mats[0], [0.95])[0])
    assert np.allclose(rb.heatmapScale(inp, "common", 0.5), [q95, q95])
    assert np.allclose(rb.heatmapScale(inp, "each", 1.0), [q95, 2 * q95])
    sparse = np.zeros((100, 10))
    sparse[0, :3] = [4.0, 5.0, 6.0]                      # 0.95 .. 0.99 quantiles are 0: ladder climbs
    want = [q for q in O.r_quantile7(sparse, [0.95, 0.96, 0.97, 0.98, 0.99, 0.995, 0.999]) if q != 0][0]
    assert np.allclose(rb.heatmapScale([{"profile": sparse}], "each"), [want])
    bad = mats[1].copy()
    bad[0, 0] = np.nan
    with pytest.raises(rb.RecoupError) as ei:
        rb.matrixQuantile(bad, [0.5])
    assert ei.value.code == _lib.RCP_ERR_DATA
    # a row block of a wider matrix: leading dimension > rows, straight through the C ABI
    big = np.asfortranarray(mats[0])
    n = 500
    out = np.empty(big.shape[1])
    sp = np.empty(big.shape[1])
    _lib.check(_lib.lib.rcp_matrix_col_profile(big.ctypes.data_as(C.c_void_p), n, big.shape[1],
                                               big.shape[0], 0, 0, _lib.MEM_HOST,
                                               out.ctypes.data_as(C.c_void_p), sp.ctypes.data_as(C.c_void_p)))
    want = O.plot_profile(big[:n], "mean")
    assert np.allclose(out, want["profile"], rtol=1e-12) and np.allclose(out + sp, want["upper"], rtol=1e-12)


def test_consumers_on_the_fixture_profile(gpu_auto, fixture_data):
    """end to end: fixture reads -> coverage -> profile -> curve, order, colour limit"""
    rb = gpu_auto
    _, g_reads = fixture_reads(fixture_data, 0)
    _, g_genes = fixture_genes(fixture_data)
    sample = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRef(sample, g_genes, "tss", (2000, 2000))
    rb.profileMatrix(sample, (2000, 2000), dict(flankBinSize=0, regionBinSize=100, sumStat="mean",
                                                 interpolation="auto"))
    m = np.asarray(sample[0]["profile"])
    curve = rb.calcPlotProfiles(sample, {"plotParams": {"sumStat": "mean", "signalScale": "natural"}})[0]
    assert np.allclose(curve["profile"], O.plot_profile(m)["profile"], rtol=1e-12)
    got = rb.orderProfiles(sample, {"orderBy": {"what": "sum1", "order": "descending"}})
    assert got["ix"].tolist() == O.r_sort_index(O.row_order_values(m, "sum"), True).tolist()
    assert np.allclose(rb.heatmapScale(sample, "common"), O.r_quantile7(m, [0.95]))


# ------------------------------------------------------------------------------------------------
# the index sort, directly
# ------------------------------------------------------------------------------------------------
def _gpu_sort(keys, bits):
    from recoup_b200 import _lib
    a = np.ascontiguousarray(keys, dtype=np.uint32).copy()
    _lib.check(_lib.lib.rcp_sort_keys_u32(a.ctypes.data_as(C.c_void_p), a.shape[0], bits, _lib.MEM_HOST))
    return a


@pytest.mark.parametrize("n,bits", [(1, 32), (2, 32), (1000, 32), (32768, 32), (32769, 32),
                                    (100_000, 27), (1_000_003, 32), (3_000_000, 17), (5_000_000, 32)])
def test_index_sort_uniform_keys(gpu, n, bits):
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << bits, size=n, dtype=np.uint64).astype(np.uint32)
    assert np.array_equal(_gpu_sort(keys, bits), np.sort(keys))


def test_index_sort_pileups_and_recursion(gpu):
    """Pile-ups: one value repeated 400 K times, 150 K keys inside a 512-wide window, 90 K inside a
    40 K-wide window, sorted / reversed inputs, all-equal input, keys of 2 significant bits."""
    rng = np.random.default_rng(5)
    parts = [np.full(400_000, 2_000_000_123, dtype=np.uint32),
             (3_000_000_000 + rng.integers(0, 512, size=150_000)).astype(np.uint32),
             (1_000_000 + rng.integers(0, 40_000, size=90_000)).astype(np.uint32),
             rng.integers(0, 1 << 32, size=1_200_000, dtype=np.uint64).astype(np.uint32),
             np.array([0, 0, 0xFFFFFFFF, 0xFFFFFFFF, 1, 0xFFFFFFFE], dtype=np.uint32)]
    keys = np.concatenate(parts)
    rng.shuffle(keys)
    want = np.sort(keys)
    assert np.array_equal(_gpu_sort(keys, 32), want)
    assert np.array_equal(_gpu_sort(want, 32), want)
    assert np.array_equal(_gpu_sort(want[::-1], 32), want)
    same = np.full(200_000, 77, dtype=np.uint32)
    assert np.array_equal(_gpu_sort(same, 32), same)
    small_range = rng.integers(0, 3, size=500_000).astype(np.uint32)      # 2 significant bits
    assert np.array_equal(_gpu_sort(small_range, 2), np.sort(small_range))


# ------------------------------------------------------------------------------------------------
# $coverage as run-length encodings (contract T1: integer Rle per region)
# ------------------------------------------------------------------------------------------------
def _np_rle(x):
    x = np.asarray(x)
    heads = np.flatnonzero(np.concatenate([[True], x[1:] != x[:-1]]))
    return x[heads].astype(np.int32), np.diff(np.concatenate([heads, [x.shape[0]]])).astype(np.int32)


def test_coverage_rle_matches_the_oracle(gpu, fixture_data):
    rb = gpu
    rng = np.random.default_rng(41)
    clen = [50000, 9000]
    chrom, s, e, st = synth_reads(rng, 6000, clen, width=(1, 300))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    rc, rs, re_, rst = _regions(rng, 150, clen, [1, 2, 255, 256, 257, 1000, 1024, 5000, 20000])
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    want = O.calc_coverage(o_reads, o_mask)
    cov = rb.calcCoverage(g_reads, g_mask)
    got = cov.rle()
    assert len(got) == len(want)
    for g, w in zip(got, want):
        if w is None:
            assert g is None
            continue
        wv, wl = _np_rle(w)
        assert np.array_equal(g[0], wv) and np.array_equal(g[1], wl)
        assert int(g[1].sum()) == w.shape[0] and (g[1] > 0).all()
    # a sub-range, and the bundled fixture (long runs of zeros between reads)
    sub = cov.rle(10, 25)
    for g, w in zip(sub, want[10:35]):
        assert (g is None) == (w is None)
        if w is not None:
            assert np.array_equal(np.repeat(g[0], g[1]), w)
    o_reads, g_reads = fixture_reads(fixture_data, 0)
    o_genes, g_genes = fixture_genes(fixture_data)
    inp = [dict(id="s", name="s", ranges=g_reads)]
    rb.coverageRef(inp, g_genes, "genebody", (2000, 2000))
    want = O.coverage_ref(o_reads, o_genes, "genebody", (2000, 2000))
    for g, w in zip(inp[0]["coverage"].rle(), want):
        assert (g is None) == (w is None)
        if w is not None:
            wv, wl = _np_rle(w)
            assert np.array_equal(g[0], wv) and np.array_equal(g[1], wl)


# ------------------------------------------------------------------------------------------------
# BASELINE.json's named configs (workloads.py generators): C2 at FULL size, C3-C5 scaled so that
# the C oracle finishes in seconds.  Coverage bit-exact (compared as dense arrays), matrices
# within 1e-6 relative, plus a checksum of checksums at full size.
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu_auto():
    import recoup_b200 as rb
    rb.init(0)
    rb.set_coverage_path("auto")
    return rb


def _dense_equal(cov, dense):
    """device CoverageList vs oracle DenseCoverage without python lists (large sizes)"""
    lens = cov.lengths().astype(np.int64)
    assert np.array_equal(lens, dense.len.astype(np.int64))
    total = int(lens.sum())
    buf = np.zeros(max(total, 1), dtype=np.int32)
    from recoup_b200 import _lib
    _lib.check(_lib.lib.rcp_coverage_fetch(cov.handle, 0, len(cov), buf.ctypes.data_as(C.POINTER(C.c_int32)),
                                           total))
    pos = 0
    off = dense.off
    for r in range(len(cov)):
        L = int(lens[r])
        if L:
            assert np.array_equal(buf[pos:pos + L], dense.cov[off[r]:off[r] + L]), "region %d" % r
            pos += L


@pytest.mark.parametrize("name,scale", [("C2", 1.0), ("C3", 0.2), ("C5", 0.1)])
def test_named_config_against_c_oracle(gpu_auto, name, scale):
    import workloads as W
    rb = gpu_auto
    w = W.CONFIGS[name](scale=scale, seed=4242)
    reads = rb.GRanges(w["read_chrom"], w["read_start"], w["read_end"], strand=w["read_strand"],
                       seqlevels=w["chrom_names"], seqlengths=w["chrom_len"])
    s, e = O.get_regional_ranges(w["region_start"], w["region_end"], w["region_strand"], w["region"],
                                 w["flank"])
    mask = rb.GRanges(w["region_chrom"], s, e, strand=w["region_strand"], seqlevels=w["chrom_names"])
    cov = rb.calcCoverage(reads, mask, frag_len=w["frag_len"])
    ix = CO.Index(w["read_chrom"], w["read_start"], w["read_end"], w["read_strand"], w["chrom_len"],
                  frag_len=w["frag_len"])
    dense = CO.coverage(ix, w["region_chrom"], s, e, w["region_strand"])
    assert cov.n_null == int((dense.len == 0).sum())
    _dense_equal(cov, dense)
    inp = [dict(id="s", name="s", coverage=cov)]
    rb.profileMatrix(inp, w["flank"], w["bin_params"])
    lens = dense.len[dense.len > 0]
    equal = bool((lens == lens[0]).all()) if lens.size else True
    want = CO.profile_matrix(dense, w["flank"], w["bin_params"], equal)
    m = np.asarray(inp[0]["profile"])
    assert_matrix_close(m, want)
    if equal and w["bin_params"]["regionBinSize"] and lens.size:
        # checksum of checksums: sum over the matrix * bases per bin == sum of all coverage
        per_bin = int(lens[0]) // int(w["bin_params"]["regionBinSize"])
        if per_bin * int(w["bin_params"]["regionBinSize"]) == int(lens[0]):
            assert abs(m.sum() * per_bin - float(dense.cov.sum(dtype=np.int64))) <= 1e-9 * max(1.0, float(dense.cov.sum(dtype=np.int64)))


def test_named_config_c4_rna_against_c_oracle(gpu_auto):
    import workloads as W
    rb = gpu_auto
    w = W.CONFIGS["C4"](scale=0.1, seed=4244)
    reads = rb.GRanges(w["read_chrom"], w["read_start"], w["read_end"], strand=w["read_strand"],
                       seqlevels=w["chrom_names"], seqlengths=w["chrom_len"])
    genes = rb.GRanges(w["region_chrom"], w["region_start"], w["region_end"], strand=w["region_strand"],
                       seqlevels=w["chrom_names"])
    grl = rb.GRangesList(rb.GRanges(w["exon_chrom"], w["exon_start"], w["exon_end"],
                                    strand=w["exon_strand"], seqlevels=w["chrom_names"]), w["exon_ptr"])
    inp = [dict(id="s", name="s", ranges=reads)]
    rb.coverageRnaRef(inp, grl, genes, w["flank"])
    ix = CO.Index(w["read_chrom"], w["read_start"], w["read_end"], w["read_strand"], w["chrom_len"])
    f1, f2 = w["flank"]
    ls, le = O.get_flanking_ranges(w["region_start"], w["region_end"], w["region_strand"], f1, "upstream")
    rs, re_ = O.get_flanking_ranges(w["region_start"], w["region_end"], w["region_strand"], f2, "downstream")
    center = CO.coverage_list(ix, w["exon_ptr"], w["exon_chrom"], w["exon_start"], w["exon_end"],
                              w["exon_strand"])
    left = CO.coverage(ix, w["region_chrom"], ls, le, w["region_strand"])
    right = CO.coverage(ix, w["region_chrom"], rs, re_, w["region_strand"])
    merged = CO.concat3(left.to_list(), center.to_list(), right.to_list())
    assert_coverage_equal(inp[0]["coverage"].to_list(), merged)
    rb.profileMatrix(inp, w["flank"], w["bin_params"])
    assert_matrix_close(inp[0]["profile"], O.profile_matrix(merged, w["flank"], w["bin_params"]))


def test_rows_scatter_places_a_row_block(gpu):
    """rcp_rows_scatter (multi-GPU helper): dst[row_index[i], c] = src[i, c], column-major."""
    import torch
    from recoup_b200 import _lib
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3)
    n_rows, n_cols, total = 1000, 37, 5000
    src = torch.from_numpy(rng.random((n_cols, n_rows + 11)))[:, :].to(dev)     # ld_src = n_rows + 11
    ids_np = rng.permutation(total)[:n_rows].astype(np.int64)
    ids = torch.from_numpy(ids_np).to(dev)
    dst = torch.zeros((n_cols, total), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    _lib.check(_lib.lib.rcp_rows_scatter(C.c_void_p(src.data_ptr()), n_rows + 11, n_rows, n_cols,
                                         C.c_void_p(ids.data_ptr()), C.c_void_p(dst.data_ptr()), total))
    _lib.check(_lib.lib.rcp_sync())
    want = np.zeros((n_cols, total))
    want[:, ids_np] = src.cpu().numpy()[:, :n_rows]
    assert np.array_equal(dst.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------
# rcp_coverage_profile: coverage -> bins without materialising the coverage
# ------------------------------------------------------------------------------------------------
def _equal_windows(rng, n, clen, L):
    chrom = rng.integers(0, len(clen), size=n).astype(np.int32)
    start = (rng.random(n) * (np.asarray(clen)[chrom] + 200)).astype(np.int64) - 100
    strand = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=n)
    return chrom, start, start + L - 1, strand


@pytest.mark.parametrize("L,n_bins", [(4000, 100), (10000, 200), (2999, 64), (900, 37), (1024, 1024),
                                      (1025, 10), (5000, 3), (300, 0)])
@pytest.mark.parametrize("ignore,filt", [(True, None), (False, None), (True, "-")])
def test_fused_coverage_profile_matches_the_oracle(gpu, L, n_bins, ignore, filt):
    """bit-exact integer sums + the same fp64 divide: the fused matrix equals profileMatrix of the
    oracle's coverage within 1e-6 (and the two-stage CUDA path exactly); NULL rows are zero and
    flagged; '-' windows are reversed; bins straddle the 896-output tiles for most sizes."""
    rb = gpu
    rng = np.random.default_rng(100 + L + n_bins)
    clen = [60000, 25000, 8000]
    chrom, s, e, st = synth_reads(rng, 30000, clen, width=(20, 300))
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    rc, rs, re_, rst = _equal_windows(rng, 400, clen, L)
    o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    filt_code = None if filt is None else {"+": 1, "-": -1, "*": 0}[filt]
    want_cov = O.calc_coverage(o_reads, o_mask, filt_code, ignore)
    bp = dict(flankBinSize=0, regionBinSize=n_bins, sumStat="mean", interpolation="auto")
    want = 0.5 * O.profile_matrix(want_cov, (0, 0), bp)
    got, is_null = rb.coverageProfile(g_reads, g_mask, n_bins, strand=filt, ignore_strand=ignore, scale=0.5)
    assert [bool(x) for x in is_null] == [w is None for w in want_cov]
    assert any(w is None for w in want_cov) and sum(w is not None for w in want_cov) > 100
    assert_matrix_close(got, want)
    # and exactly what the two stages give
    cov = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
    cov.set_scale(0.5)
    inp = [dict(id="s", name="s", ranges=g_reads, coverage=cov)]
    rb.profileMatrix(inp, (0, 0), bp)
    assert np.array_equal(np.asarray(got), np.asarray(inp[0]["profile"]))


def test_fused_coverage_profile_device_memory_and_errors(gpu):
    import torch
    from recoup_b200 import _lib
    rb = gpu
    L = _lib.lib
    rng = np.random.default_rng(5)
    clen = [50000, 20000]
    chrom, s, e, st = synth_reads(rng, 20000, clen, width=(30, 200))
    _, g_reads = both_reads(chrom, s, e, st, clen)
    rc, rs, re_, rst = _equal_windows(rng, 300, clen, 3000)
    _, g_mask = both_regions(rc, rs, re_, rst, len(clen))
    want, want_null = rb.coverageProfile(g_reads, g_mask, 60)
    dr = rb.device_reads(g_reads)
    dev = torch.device("cuda", 0)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)      # noqa: E731
    d = [t(g_mask.seqnames, np.int32), t(g_mask.start, np.int32), t(g_mask.end, np.int32), t(g_mask.strand, np.int8)]
    out = torch.full((60, 300 + 7), -1.0, dtype=torch.float64, device=dev)          # ld = 307 > n_regions
    nul = torch.full((300,), 9, dtype=torch.uint8, device=dev)
    vp = lambda x: C.c_void_p(x.data_ptr())                                          # noqa: E731
    _lib.check(L.rcp_coverage_profile(dr.handle, 300, vp(d[0]), vp(d[1]), vp(d[2]), vp(d[3]), 1, _lib.STRAND_ANY,
                                      60, 42, 0, 1.0, vp(out), 307, vp(nul), _lib.MEM_DEVICE))
    L.rcp_sync()
    got = out.cpu().numpy()
    assert np.array_equal(got[:, :300].T, np.asarray(want))
    assert (got[:, 300:] == -1.0).all()                      # the padding rows of ld are untouched
    assert np.array_equal(nul.cpu().numpy().astype(bool), want_null)
    # windows of different lengths: an error, not a silently binned mixture
    re2 = re_.copy()
    re2[7] += 5
    _, bad_mask = both_regions(rc, rs, re2, rst, len(clen))
    with pytest.raises(rb.RecoupError):
        rb.coverageProfile(g_reads, bad_mask, 60)
    # windows shorter than the bin count take the composed path (spline / neighbourhood fill)
    rc3, rs3, re3, rst3 = _equal_windows(rng, 50, clen, 40)
    o3, m3 = both_regions(rc3, rs3, re3, rst3, len(clen))
    o_reads, _ = both_reads(chrom, s, e, st, clen)
    got3, _ = rb.coverageProfile(g_reads, m3, 64)
    bp = dict(flankBinSize=0, regionBinSize=64, sumStat="mean", interpolation="auto")
    assert_matrix_close(got3, O.profile_matrix(O.calc_coverage(o_reads, o3, None, True), (0, 0), bp))


def test_auto_serves_ordinary_samples_through_the_split_path(gpu_auto):
    """RCP_PATH_AUTO: short reads over a GRanges mask go through the one-pass split path; reads
    wider than its packed word allows take the buckets (same results either way).  The retired
    RCP_PATH_BLOCKS selects the buckets too."""
    from recoup_b200 import _lib
    rb = gpu_auto
    rng = np.random.default_rng(8)
    clen = [90000, 30000]

    def path_of(cov):
        pth, cand = C.c_int(0), C.c_int64(0)
        _lib.check(_lib.lib.rcp_coverage_path_info(cov.handle, C.byref(pth), C.byref(cand)))
        return pth.value, cand.value

    for width, want_path in (((30, 250), 4), ((9000, 12000), 2)):
        chrom, s, e, st = synth_reads(rng, 5000, clen, width=width)
        o_reads, g_reads = both_reads(chrom, s, e, st, clen)
        rc, rs, re_, rst = _equal_windows(rng, 100, clen, 2500)
        o_mask, g_mask = both_regions(rc, rs, re_, rst, len(clen))
        want = O.calc_coverage(o_reads, o_mask, None, True)
        cov = rb.calcCoverage(g_reads, g_mask)
        pth, cand = path_of(cov)
        assert pth == want_path
        if want_path == 4:
            assert cand > 0
        assert_coverage_equal(cov.to_list(), want)
    rb.set_coverage_path("blocks")
    try:
        cov = rb.calcCoverage(g_reads, g_mask)
    finally:
        rb.set_coverage_path("auto")
    assert path_of(cov)[0] == 2
    assert_coverage_equal(cov.to_list(), want)


def test_region_sharded_run_equals_the_single_gpu_matrix(gpu_auto):
    """The multi-GPU path with the CUDA library behind every rank, emulated in one process (the
    ranks of a box run the same code on their own GPUs): partition_regions + slice_spans +
    exchange_reads (world 1: the local filter) per slice, the row blocks put back by row index --
    bitwise equal to the one-GPU matrix, coverage included."""
    import torch
    import workloads as W
    from recoup_b200.sharding import exchange_reads, partition_regions, slice_spans
    rb = gpu_auto
    w = W.dnase_sites(scale=0.002, seed=17)
    genes = rb.GRanges(w["region_chrom"], w["region_start"], w["region_end"], strand=w["region_strand"],
                       seqlevels=w["chrom_names"])
    win = rb.getRegionalRanges(genes, "custom", w["flank"])
    reads = rb.GRanges(w["read_chrom"], w["read_start"], w["read_end"], strand=w["read_strand"],
                       seqlevels=w["chrom_names"], seqlengths=w["chrom_len"])
    full, _ = rb.coverageProfile(reads, win, 0)
    full_cov = rb.calcCoverage(reads, win).to_list()
    world = 3
    parts = partition_regions(win.seqnames, win.start, win.end, world)
    spans = slice_spans(win.seqnames, win.start, win.end, parts, len(w["chrom_len"]))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))      # noqa: E731
    got = np.full_like(np.asarray(full), -1.0)
    for rank in range(world):
        idx = np.sort(parts[rank])
        # world 1 inside exchange_reads: the local filter against THIS rank's spans
        c, s, e, st = exchange_reads(t(w["read_chrom"]), t(w["read_start"]), t(w["read_end"]), t(w["read_strand"]),
                                     spans[rank:rank + 1])
        assert 0 < c.shape[0] < len(w["read_start"])
        mine = rb.GRanges(c.numpy(), s.numpy(), e.numpy(), strand=st.numpy(), seqlevels=w["chrom_names"],
                          seqlengths=w["chrom_len"])
        block, _ = rb.coverageProfile(mine, win.subset(idx), 0)
        got[idx] = np.asarray(block)
        cov = rb.calcCoverage(mine, win.subset(idx)).to_list()
        for k, i in enumerate(idx):
            a, b = cov[k], full_cov[int(i)]
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
    assert np.array_equal(got, np.asarray(full))


@pytest.mark.parametrize("n_reads", [1, 2047, 50000])
def test_read_routing_kernels_match_the_span_rule(gpu_auto, n_reads):
    """rcp_reads_route_count / _pack (the send side of the region-sharded exchange): rank r's run
    holds exactly the reads that meet r's spans (a boundary read goes to both neighbours, a read
    with a bad chromosome id to rank 0), strands travel with their reads; and exchange_reads on
    device tensors (world 1) returns the same reads as on host tensors."""
    import torch
    from recoup_b200 import _lib
    from recoup_b200.sharding import exchange_reads, partition_regions, slice_spans
    rng = np.random.default_rng(23)
    clen = [90000, 30000, 5000]
    chrom, s, e, st = synth_reads(rng, n_reads, clen, width=(20, 400))
    if n_reads > 10:
        chrom[3] = 7                                         # outside the table: rank 0 reports it
    rc, rs, re_, rst = _regions(rng, 90, clen, [100, 1000, 3000])
    world = 3
    parts = partition_regions(rc, rs, re_, world)
    spans = slice_spans(rc, rs, re_, parts, len(clen))
    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (chrom, s.astype(np.int32), e.astype(np.int32), st)]
    vp = lambda t: C.c_void_p(t.data_ptr())                  # noqa: E731
    sp = np.ascontiguousarray(np.clip(spans, -2**31 + 1, 2**31 - 1), dtype=np.int32)
    sp_p = sp.ctypes.data_as(C.POINTER(C.c_int32))
    counts = np.zeros(world, dtype=np.int64)
    L = _lib.lib
    _lib.check(L.rcp_reads_route_count(n_reads, vp(d[0]), vp(d[1]), vp(d[2]), world, len(clen), sp_p,
                                       counts.ctypes.data_as(C.POINTER(C.c_int64))))
    ok = (chrom >= 0) & (chrom < len(clen))
    cc = np.where(ok, chrom, 0)
    want = []
    for r in range(world):
        m = ok & (e >= spans[r, cc, 0]) & (s <= spans[r, cc, 1])
        if r == 0:
            m |= ~ok
        want.append(np.flatnonzero(m))
    assert counts.tolist() == [len(x) for x in want]
    offsets = np.concatenate(([0], np.cumsum(counts)[:-1])).astype(np.int64)
    total = int(counts.sum())
    outs = [torch.full((max(total, 1),), -9, dtype=torch.int32, device=dev) for _ in range(3)]
    so = torch.full((max(total, 1),), -9, dtype=torch.int8, device=dev)
    _lib.check(L.rcp_reads_route_pack(n_reads, vp(d[0]), vp(d[1]), vp(d[2]), vp(d[3]), world, len(clen), sp_p,
                                      offsets.ctypes.data_as(C.POINTER(C.c_int64)), vp(outs[0]), vp(outs[1]),
                                      vp(outs[2]), vp(so)))
    L.rcp_sync()
    tri, so = np.column_stack([o.cpu().numpy() for o in outs]), so.cpu().numpy()
    for r in range(world):
        got = np.column_stack([tri[offsets[r]:offsets[r] + counts[r]], so[offsets[r]:offsets[r] + counts[r]]])
        exp = np.column_stack([chrom[want[r]], s[want[r]], e[want[r]], st[want[r]]])
        assert np.array_equal(got[np.lexsort(got.T[::-1])], exp[np.lexsort(exp.T[::-1])])
    # the wrapper, device tensors against host tensors (world 1: the local filter against rank 1's spans)
    if n_reads > 10:
        keep = ok
        dk = [torch.from_numpy(np.ascontiguousarray(a[keep])) for a in (chrom, s.astype(np.int32), e.astype(np.int32), st)]
        host = exchange_reads(*dk, spans[1:2])
        stream = torch.cuda.ExternalStream(L.rcp_stream(), device=dev)
        with torch.cuda.stream(stream):
            devr = exchange_reads(*[t.to(dev) for t in dk], spans[1:2])
        L.rcp_sync()
        a = np.column_stack([t.cpu().numpy() for t in devr])
        b = np.column_stack([t.numpy() for t in host])
        assert np.array_equal(a[np.lexsort(a.T[::-1])], b[np.lexsort(b.T[::-1])])


@pytest.mark.parametrize("ignore,filt", [(True, None), (False, None), (False, "+")])
def test_list_masks_with_long_reads_and_the_cached_binned_index(gpu, ignore, filt):
    """GRangesList elements over a sample that mixes short reads with reads far wider than the
    packed candidate word (unspliced / long reads, 2 %): the first list call builds the handle's
    binned index (short reads) + long-read list, and the GRanges calls that follow on the SAME
    handle (coverageRnaRef's flank passes) reuse both.  Multiplicity of long reads spanning
    several exons included."""
    rb = gpu
    rng = np.random.default_rng(77)
    clen = [150000, 40000]
    chrom, s, e, st = synth_reads(rng, 30000, clen, width=(30, 300))
    lc, ls, le, lst = synth_reads(rng, 600, clen, width=(9000, 30000))
    chrom, s, e, st = (np.concatenate([chrom, lc]), np.concatenate([s, ls]), np.concatenate([e, le]),
                       np.concatenate([st, lst]))
    perm = rng.permutation(chrom.shape[0])
    chrom, s, e, st = chrom[perm], s[perm], e[perm], st[perm]
    o_reads, g_reads = both_reads(chrom, s, e, st, clen)
    ptr, xc, xs, xe, xst = [0], [], [], [], []
    for g in range(120):
        c = int(rng.integers(0, 2))
        pos = int(rng.integers(1, clen[c] - 30000))
        gst = int(rng.choice([1, -1, 0]))
        for _ in range(int(rng.integers(1, 14))):
            w = int(rng.integers(20, 900))
            xc.append(c); xs.append(pos); xe.append(pos + w - 1); xst.append(gst)
            pos += w + int(rng.integers(50, 2500))
        ptr.append(len(xs))
    o_mask = dict(ptr=ptr, chrom=xc, start=xs, end=xe, strand=xst)
    u = rb.GRanges(np.asarray(xc, np.int32), xs, xe, strand=np.asarray(xst, np.int8), seqlevels=["c0", "c1"])
    g_mask = rb.GRangesList(u, ptr)
    filt_code = None if filt is None else {"+": 1, "-": -1, "*": 0}[filt]
    want = O.calc_coverage(o_reads, o_mask, filt_code, ignore)
    got = rb.calcCoverage(g_reads, g_mask, strand=filt, ignore_strand=ignore)
    assert_coverage_equal(got.to_list(), want)
    # the GRanges passes that follow on the same handle
    rc, rs, re_, rst = _regions(rng, 200, clen, [1, 90, 1000, 1024, 1025, 3000, 9000, 20011])
    o2, g2 = both_regions(rc, rs, re_, rst, len(clen))
    want2 = O.calc_coverage(o_reads, o2, filt_code, ignore)
    got2 = rb.calcCoverage(g_reads, g2, strand=filt, ignore_strand=ignore)
    assert_coverage_equal(got2.to_list(), want2)
    m, is_null = rb.coverageProfile(g_reads, g2.subset(np.flatnonzero(np.asarray(re_) - np.asarray(rs) == 2999)), 30,
                                    strand=filt, ignore_strand=ignore)
    sel = [w for w, L in zip(want2, np.asarray(re_) - np.asarray(rs)) if L == 2999]
    bp = dict(flankBinSize=0, regionBinSize=30, sumStat="mean", interpolation="auto")
    assert_matrix_close(m, O.profile_matrix(sel, (0, 0), bp))
