"""BigWig input: the loader (rcp_bigwig_load), signal coverage (rcp_signal_coverage) and the
profile kernels over FLOAT32 coverage, against tests/bigwig_writer.py and oracle/bigwig_oracle.py
(parity unpinned: the reference's BigWig lines cannot run here)."""
import os
import struct

import numpy as np
import pytest

from oracle import bigwig_oracle as BO
from oracle import recoup_oracle as O
from tests.bigwig_writer import items_of, write_bigwig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def bw_gpu():
    import recoup_b200 as rb
    rb.init(0)
    return rb


# ---------------------------------------------------------------------------------------------
# Hand-assembled known-answer file: two chromosomes, one stored bedGraph block, one R-tree leaf
# ---------------------------------------------------------------------------------------------
KAT_CHROMS = [("chr1", 1000), ("chr2", 500)]
KAT_ITEMS = [(0, 10, 1.5), (20, 30, -2.0), (990, 1000, 0.25)]       # chr1, 0-based half-open


def kat_bytes():
    header = struct.pack("<I", 0x888FFC26)        # magic
    header += struct.pack("<H", 4)                # version
    header += struct.pack("<H", 0)                # zoomLevels
    header += struct.pack("<Q", 64)               # chromTreeOffset
    header += struct.pack("<Q", 124)              # fullDataOffset
    header += struct.pack("<Q", 192)              # fullIndexOffset
    header += struct.pack("<H", 0)                # fieldCount
    header += struct.pack("<H", 0)                # definedFieldCount
    header += struct.pack("<Q", 0)                # autoSqlOffset
    header += struct.pack("<Q", 0)                # totalSummaryOffset
    header += struct.pack("<I", 0)                # uncompressBufSize (0: blocks stored)
    header += struct.pack("<Q", 0)                # reserved (extension offset)
    tree = struct.pack("<I", 0x78CA8C91)          # chromosome B+ tree: magic
    tree += struct.pack("<I", 2)                  # blockSize
    tree += struct.pack("<I", 4)                  # keySize
    tree += struct.pack("<I", 8)                  # valSize
    tree += struct.pack("<Q", 2)                  # itemCount
    tree += struct.pack("<Q", 0)                  # reserved
    tree += struct.pack("<BBH", 1, 0, 2)          # node: isLeaf, reserved, count
    tree += b"chr1" + struct.pack("<II", 0, 1000)  # key, chromId, chromSize
    tree += b"chr2" + struct.pack("<II", 1, 500)
    data = struct.pack("<Q", 1)                   # sectionCount
    data += struct.pack("<IIIII", 0, 0, 1000, 0, 0)   # section: chromId, start, end, itemStep, itemSpan
    data += struct.pack("<BBH", 1, 0, 3)          # type (1 bedGraph), reserved, itemCount
    for s, e, v in KAT_ITEMS:
        data += struct.pack("<IIf", s, e, v)      # chromStart, chromEnd, value
    index = struct.pack("<I", 0x2468ACE0)         # R-tree: magic
    index += struct.pack("<I", 1)                 # blockSize
    index += struct.pack("<Q", 1)                 # itemCount
    index += struct.pack("<IIII", 0, 0, 0, 1000)  # startChromIx, startBase, endChromIx, endBase
    index += struct.pack("<Q", 192)               # endFileOffset
    index += struct.pack("<II", 1024, 0)          # itemsPerSlot, reserved
    index += struct.pack("<BBH", 1, 0, 1)         # node: isLeaf, reserved, count
    index += struct.pack("<IIII", 0, 0, 0, 1000)  # startChromIx, startBase, endChromIx, endBase
    index += struct.pack("<QQ", 132, 60)          # dataOffset, dataSize
    out = header + tree + data + index
    assert len(header) == 64 and len(header + tree) == 124 and len(header + tree + data) == 192
    return out


KAT_SECTIONS = [dict(chrom=0, type="bedGraph", items=KAT_ITEMS)]


def test_writer_reproduces_the_hand_assembled_file():
    got = write_bigwig(KAT_CHROMS, KAT_SECTIONS, compress=False, chrom_block=2, rtree_block=1)
    assert got == kat_bytes()


# ---------------------------------------------------------------------------------------------
# Oracle known answers
# ---------------------------------------------------------------------------------------------
def small_track():
    # chr0 (100 bp): 1.0 on 5..10, 2.5 on 20, -1.0 on 95..100; chr1 (50 bp): no item
    return BO.Track([0, 0, 0], [5, 20, 95], [10, 20, 100], [1.0, 2.5, -1.0], [100, 50])


def one(track, c, s, e, st=1):
    return BO.coverage_from_track(track, c, [s], [e], [st])


def test_oracle_known_answers():
    t = small_track()
    v = t.chrom_vector(0)
    assert v.shape == (100,) and v[4:10].tolist() == [1.0] * 6 and v[19] == 2.5 and v[94:].tolist() == [-1.0] * 6
    assert np.array_equal(t.values_at(0, np.arange(1, 101)), v)
    assert one(t, 0, 1, 12).tolist() == [0] * 4 + [1.0] * 6 + [0, 0]            # gaps
    assert one(t, 0, 11, 19).tolist() == [0.0] * 9                               # no item: zeros, not NULL
    assert one(t, 0, 0, 3).tolist() == [0.0] * 3                                 # start 0 is dropped
    assert one(t, 0, 96, 100).tolist() == [-1.0] * 5                             # right edge
    assert one(t, 0, 98, 101) is None                                            # past chromSize
    assert one(t, 0, -1, 5) is None                                              # negative subscript
    assert one(t, 0, 18, 21, -1).tolist() == [0, 2.5, 0, 0]                      # reversed on '-'
    assert one(t, 1, 1, 50).tolist() == [0.0] * 50                               # chromosome without items
    assert one(t, -1, 1, 5) is None                                              # not in the track
    plus = BO.coverage_from_track(t, 0, [4, 19], [6, 21], [1, -1])
    assert plus.tolist() == [0, 1, 1, 0, 2.5, 0]                                 # stitched, FIRST strand
    minus = BO.coverage_from_track(t, 0, [4, 19], [6, 21], [-1, 1])
    assert minus.tolist() == [0, 2.5, 0, 1, 1, 0]
    assert BO.coverage_from_track(t, 0, [4, 99], [6, 101], [1, 1]) is None       # one range out of bounds


def test_calccoverage_bigwig_path_errors(tmp_path):
    import recoup_b200 as rb
    gr = rb.GRanges(np.zeros(1, np.int32), [1], [10], seqlevels=["c0"], seqlengths=[100])
    for name in ("missing.bw", "missing.BigWig", "MISSING.BW"):
        with pytest.raises(ValueError, match="input argument must be a GenomicRanges"):
            rb.calcCoverage(str(tmp_path / name), mask=gr)                       # coverage.R:129
    with pytest.raises(NotImplementedError):
        rb.calcCoverage(str(tmp_path / "sample.bwx"), mask=gr)


# ---------------------------------------------------------------------------------------------
# Random tracks
# ---------------------------------------------------------------------------------------------
def random_value(rng):
    r = rng.random()
    if r < 0.05:
        return 0.0
    if r < 0.08:
        return -0.0
    return float(np.float32(rng.normal(0, 20)))


def random_sections(rng, chroms, skip=()):
    """Sections of every type over each chromosome (not those in `skip`), sorted and disjoint."""
    secs = []
    for c, (_, size) in enumerate(chroms):
        if c in skip:
            continue
        pos = int(rng.integers(0, 50))
        while pos < size - 10:
            kind = rng.choice(["bedGraph", "varStep", "fixedStep"])
            n = int(rng.integers(1, 300))
            if kind == "bedGraph":
                items = []
                for _ in range(n):
                    s = pos + int(rng.integers(0, 40))
                    e = s + int(rng.integers(1, 60))
                    if e > size:
                        break
                    items.append((s, e, random_value(rng)))
                    pos = e
                if items:
                    secs.append(dict(chrom=c, type=kind, items=items))
            elif kind == "varStep":
                span = int(rng.integers(1, 30))
                items = []
                for _ in range(n):
                    s = pos + int(rng.integers(0, 40))
                    if s + span > size:
                        break
                    items.append((s, random_value(rng)))
                    pos = s + span
                if items:
                    secs.append(dict(chrom=c, type=kind, items=items, span=span))
            else:
                span = int(rng.integers(1, 30))
                step = span + int(rng.integers(0, 10))
                n = max(1, min(n, (size - pos - span) // step + 1))
                if pos + span > size:
                    break
                secs.append(dict(chrom=c, type=kind, start=pos, step=step, span=span,
                                 items=[random_value(rng) for _ in range(n)]))
                pos += (n - 1) * step + span
            pos += int(rng.integers(0, 2000))               # a gap between sections
    return secs


TRACK_CHROMS = [("chrA", 30000), ("chrB", 45000), ("chrC", 20000), ("chrD", 12000), ("chrE", 9000)]
MASK_LEVELS = ["chrB", "chrA", "chrX", "chrC", "chrE"]      # chrX: not in the track; chrD: not in the mask


def track_and_oracle(seed, compress, chrom_block=2, rtree_block=3, zoom=2):
    rng = np.random.default_rng(seed)
    secs = random_sections(rng, TRACK_CHROMS, skip=(4,))     # chrE has no item
    data = write_bigwig(TRACK_CHROMS, secs, compress=compress, chrom_block=chrom_block,
                        rtree_block=rtree_block, zoom_levels=zoom)
    oracle = BO.Track.from_file_items(items_of(secs), [s for _, s in TRACK_CHROMS])
    return data, oracle, secs


def random_windows(rng, n):
    sizes = {n_: s for n_, s in TRACK_CHROMS}
    sizes["chrX"] = 10000
    lv = rng.integers(0, len(MASK_LEVELS), size=n)
    start, end = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for i in range(n):
        size = sizes[MASK_LEVELS[lv[i]]]
        kind = rng.integers(0, 8)
        w = int(rng.integers(1, 3000))
        if kind == 0:
            s = 1
        elif kind == 1:
            s = size - w + 1
        elif kind == 2:
            s = size - w + 5                                # past the end -> NULL
        elif kind == 3:
            s = 0                                            # a 0 subscript is dropped
        elif kind == 4:
            s = -int(rng.integers(1, 10))                    # negative -> NULL
        else:
            s = int(rng.integers(1, max(size - w, 2)))
        start[i], end[i] = s, s + w - 1
    strand = rng.choice(np.array([1, -1, 0], dtype=np.int8), size=n)
    return lv, start, end, strand


def oracle_mask(lv, start, end, strand, ptr=None):
    track_ids = {n: i for i, (n, _) in enumerate(TRACK_CHROMS)}
    chrom = np.asarray([track_ids.get(MASK_LEVELS[c], -1) for c in lv], dtype=np.int64)
    m = dict(chrom=chrom, start=start, end=end, strand=np.asarray(strand, np.int64))
    if ptr is not None:
        m["ptr"] = ptr
    return m


def assert_signal_equal(got, want):
    """Signal coverage parity is BIT-EXACT (float32 words)."""
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        if w is None:
            assert g is None, "element %d: oracle NULL, CUDA length %d" % (i, len(g))
            continue
        assert g is not None, "element %d: CUDA NULL, oracle length %d" % (i, len(w))
        assert g.dtype == np.float32 and g.shape == w.shape, (i, g.dtype, g.shape, w.shape)
        assert np.array_equal(g.view(np.uint32), w.view(np.uint32)), "element %d differs" % i


def runs_of(v):
    b = v.view(np.uint32)
    head = np.concatenate([[True], b[1:] != b[:-1]])
    starts = np.flatnonzero(head)
    return v[starts], np.diff(np.concatenate([starts, [v.shape[0]]])).astype(np.int32)


@pytest.mark.gpu
def test_kat_items_fetch_exactly(bw_gpu):
    rb = bw_gpu
    t = rb.readBigWig(kat_bytes())
    assert t.seqlevels == ["chr1", "chr2"] and t.seqlengths.tolist() == [1000, 500] and len(t) == 3
    chrom, start, end, value = t.fetch()
    assert chrom.tolist() == [0, 0, 0]
    assert start.tolist() == [1, 21, 991] and end.tolist() == [10, 30, 1000]
    assert value.tolist() == [1.5, -2.0, 0.25]
    t.free()


@pytest.mark.gpu
@pytest.mark.parametrize("compress", [True, False])
@pytest.mark.parametrize("seed", [1, 2])
def test_random_tracks_coverage_and_rle_bit_exact(bw_gpu, compress, seed):
    rb = bw_gpu
    data, oracle, secs = track_and_oracle(seed, compress)
    t = rb.readBigWig(data, threads=3)
    want_items = sorted((c, s + 1, e, np.float32(v) + np.float32(0)) for c, s, e, v in items_of(secs))
    chrom, start, end, value = t.fetch()
    assert len(t) == len(want_items)
    assert chrom.tolist() == [x[0] for x in want_items] and start.tolist() == [x[1] for x in want_items]
    assert end.tolist() == [x[2] for x in want_items]
    assert np.array_equal(value.view(np.uint32), np.asarray([x[3] for x in want_items], np.float32).view(np.uint32))
    rng = np.random.default_rng(seed + 100)
    lv, s, e, st = random_windows(rng, 400)
    mask = rb.GRanges(lv.astype(np.int32), s, e, strand=st, seqlevels=MASK_LEVELS)
    got = rb.calcCoverage(t, mask)
    want = BO.calc_coverage(oracle, oracle_mask(lv, s, e, st))
    assert got.dtype == np.float32
    assert any(w is None for w in want) and any(w is not None and not w.any() for w in want)
    assert_signal_equal(got.to_list(), want)
    for g, w in zip(got.rle(), want):
        if w is None:
            assert g is None
        else:
            wv, wl = runs_of(w)
            assert np.array_equal(g[0].view(np.uint32), wv.view(np.uint32)) and np.array_equal(g[1], wl)
    # calcCoverage also takes a path ending in .bw
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), "rcp_test_%d_%d_%d.bw" % (os.getpid(), seed, compress))
    with open(path, "wb") as f:
        f.write(data)
    try:
        assert_signal_equal(rb.calcCoverage(path, mask).to_list(), want)
    finally:
        os.unlink(path)
    t.free()


def random_gene_list(rng, n_genes):
    """GRangesList of exons (several per gene, on the chromosome of the first) + the genes."""
    sizes = {n_: s for n_, s in TRACK_CHROMS}
    sizes["chrX"] = 10000
    lv, s, e, st, ptr = [], [], [], [], [0]
    g_lv, g_s, g_e, g_st = [], [], [], []
    for _ in range(n_genes):
        c = int(rng.integers(0, len(MASK_LEVELS)))
        size = sizes[MASK_LEVELS[c]]
        k = int(rng.integers(1, 6))
        pos = int(rng.integers(2000, max(size - 8000, 2001)))
        strand = int(rng.choice([1, -1]))
        first = pos
        for _ in range(k):
            a = pos + int(rng.integers(0, 300))
            b = a + int(rng.integers(0, 400))
            lv.append(c), s.append(a), e.append(b), st.append(strand)
            pos = b + 1
        ptr.append(len(s))
        g_lv.append(c), g_s.append(first), g_e.append(pos), g_st.append(strand)
    return (np.asarray(lv), np.asarray(s), np.asarray(e), np.asarray(st, np.int8), np.asarray(ptr, np.int64),
            np.asarray(g_lv), np.asarray(g_s), np.asarray(g_e), np.asarray(g_st, np.int8))


@pytest.mark.gpu
def test_granges_list_and_coverage_rna_ref(bw_gpu, tmp_path):
    rb = bw_gpu
    data, oracle, _ = track_and_oracle(5, True)
    rng = np.random.default_rng(55)
    lv, s, e, st, ptr, g_lv, g_s, g_e, g_st = random_gene_list(rng, 150)
    u = rb.GRanges(lv.astype(np.int32), s, e, strand=st, seqlevels=MASK_LEVELS)
    names = ["g%d" % i for i in range(len(ptr) - 1)]
    grl = rb.GRangesList(u, ptr, names=names)
    t = rb.readBigWig(data)
    want_center = BO.calc_coverage(oracle, oracle_mask(lv, s, e, st, ptr))
    assert_signal_equal(rb.calcCoverage(t, grl).to_list(), want_center)
    t.free()
    genes = rb.GRanges(g_lv.astype(np.int32), g_s, g_e, strand=g_st, seqlevels=MASK_LEVELS, names=names)
    path = str(tmp_path / "track.bigWig")
    with open(path, "wb") as f:
        f.write(data)
    inp = [dict(id="bw", name="bw", file=path, format="bigwig", ranges=None)]
    rb.coverageRnaRef(inp, grl, genes, (700, 500))
    parts = []
    for side, w in (("upstream", 700), ("downstream", 500)):
        ls, le = O.get_flanking_ranges(g_s, g_e, g_st, w, side)
        parts.append(BO.calc_coverage(oracle, oracle_mask(g_lv, ls, le, g_st)))
    want = [None if a is None or b is None or c is None else np.concatenate([a, b, c])
            for a, b, c in zip(parts[0], want_center, parts[1])]
    assert any(w is not None for w in want)
    assert_signal_equal(inp[0]["coverage"].to_list(), want)


def assert_bins_close(got, want, absm, interp_rows=None):
    """bin means: |got - want| <= 1e-9 * mean(|x|) over the bin, exactly 0 for all-zero bins;
    rows that went through interpolation: the tolerance of the interpolation tests."""
    got, want, absm = np.asarray(got), np.asarray(want), np.asarray(absm)
    assert got.shape == want.shape
    rows = np.ones(got.shape[0], bool) if interp_rows is None else ~interp_rows
    g, w, a = got[rows], want[rows], absm[rows]
    assert np.all(np.abs(g - w) <= 1e-9 * a)
    assert np.all(g[a == 0] == 0)
    if interp_rows is not None and interp_rows.any():
        np.testing.assert_allclose(got[interp_rows], want[interp_rows], rtol=1e-6, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("stat", ["mean", "median"])
def test_profile_matrix_over_signal(bw_gpu, stat):
    rb = bw_gpu
    data, oracle, _ = track_and_oracle(7, True)
    t = rb.readBigWig(data)
    rng = np.random.default_rng(77)
    # equal-length windows (TSS +- 1 kb) -> 50 bins
    lv, s, e, st = random_windows(rng, 300)
    s = np.where(s < 1, 1, s)
    w = 2000
    mask = rb.GRanges(lv.astype(np.int32), s, s + w - 1, strand=st, seqlevels=MASK_LEVELS)
    cov = rb.calcCoverage(t, mask)
    want_cov = BO.calc_coverage(oracle, oracle_mask(lv, s, s + w - 1, st))
    assert_signal_equal(cov.to_list(), want_cov)
    bp = dict(flankBinSize=0, regionBinSize=50, sumStat=stat, interpolation="auto")
    inp = [dict(id="a", name="a", coverage=cov)]
    rb.profileMatrix(inp, (1000, 1000), bp)
    want = O.profile_matrix(want_cov, (1000, 1000), bp)
    if stat == "median":
        assert np.array_equal(np.asarray(inp[0]["profile"]), want)
    else:
        absm = O.profile_matrix([None if c is None else np.abs(c) for c in want_cov], (1000, 1000), bp)
        assert_bins_close(inp[0]["profile"], want, absm)
    # per-base matrix (exact) and set_scale
    base = rb.baseCoverageMatrix(cov, flank=(1000, 1000), where="upstream")
    assert np.array_equal(np.asarray(base), O.base_coverage_matrix(want_cov, (1000, 1000), "upstream"))
    whole = rb.baseCoverageMatrix(cov)
    assert np.array_equal(np.asarray(whole), O.base_coverage_matrix(want_cov))
    cov.set_scale(0.5)
    scaled = rb.baseCoverageMatrix(cov)
    assert np.array_equal(np.asarray(scaled), 0.5 * O.base_coverage_matrix(want_cov))
    # gene bodies with flanks; short genes take the spline / neighbourhood paths
    g_s = rng.integers(3000, 8000, size=120)
    g_len = np.concatenate([rng.integers(5, 60, size=40), rng.integers(100, 9000, size=80)])
    g_lv = rng.choice([0, 1, 3], size=120)
    g_st = rng.choice(np.array([1, -1], np.int8), size=120)
    f = (500, 300)
    gs, ge = g_s - f[0], g_s + g_len - 1 + f[1]
    gs, ge = np.where(g_st < 0, g_s - f[1], gs), np.where(g_st < 0, g_s + g_len - 1 + f[0], ge)
    mask = rb.GRanges(g_lv.astype(np.int32), gs, ge, strand=g_st, seqlevels=MASK_LEVELS)
    cov = rb.calcCoverage(t, mask)
    want_cov = BO.calc_coverage(oracle, oracle_mask(g_lv, gs, ge, g_st))
    assert_signal_equal(cov.to_list(), want_cov)
    bp = dict(flankBinSize=25, regionBinSize=64, sumStat=stat, interpolation="auto")
    inp = [dict(id="a", name="a", coverage=cov)]
    rb.profileMatrix(inp, f, bp)
    want = O.profile_matrix(want_cov, f, bp, equal_lengths=False)
    short = np.asarray([c is not None and c.shape[0] - f[0] - f[1] < 64 for c in want_cov])
    assert short.any()
    absm = O.profile_matrix([None if c is None else np.abs(c) for c in want_cov], f, bp, equal_lengths=False)
    if stat == "median":
        assert np.array_equal(np.asarray(inp[0]["profile"])[~short], want[~short])
        np.testing.assert_allclose(np.asarray(inp[0]["profile"])[short], want[short], rtol=1e-6, atol=1e-12)
    else:
        assert_bins_close(inp[0]["profile"], want, absm, interp_rows=short)
    t.free()


# ---------------------------------------------------------------------------------------------
# Data errors, one each
# ---------------------------------------------------------------------------------------------
def patched(data, at, fmt, value):
    b = bytearray(data)
    struct.pack_into(fmt, b, at, value)
    return bytes(b)


def block0(data):
    return struct.unpack_from("<Q", data, 16)[0] + 8        # fullDataOffset + sectionCount


def bad_files():
    kat = kat_bytes()
    b0 = block0(kat)
    w = lambda secs, size=1000: write_bigwig([("chr1", size), ("chr2", 500)], secs, compress=False)
    bg = lambda items: [dict(chrom=0, type="bedGraph", items=items)]
    return {
        "bad magic": (kat[:0] + b"\0\0\0\0" + kat[4:], "bad magic"),
        "bigBed": (patched(kat, 0, "<I", 0x8789F2EB), "bigBed, not bigWig"),
        "truncated": (kat[:150], "truncated"),
        "section size": (patched(kat, b0 + 22, "<H", 4), "section size"),
        "unsorted": (w(bg([(20, 30, 1.0), (0, 10, 2.0)])), "not sorted"),
        "overlap": (w(bg([(0, 10, 1.0), (9, 12, 2.0)])), "not sorted"),
        "overlap across blocks": (w(bg([(0, 10, 1.0)]) + bg([(5, 12, 2.0)])), "not sorted"),
        "end <= start": (w(bg([(10, 10, 1.0)])), "end <= start"),
        "past chromSize": (w(bg([(990, 1001, 1.0)])), "past chromSize"),
        "nan": (w(bg([(0, 10, float("nan"))])), "NaN or infinite"),
        "inf": (w(bg([(0, 10, float("-inf"))])), "NaN or infinite"),
    }


@pytest.mark.gpu
def test_every_data_error(bw_gpu):
    rb = bw_gpu
    from recoup_b200 import _lib
    for name, (data, msg) in bad_files().items():
        with pytest.raises(rb.RecoupError, match=msg) as ei:
            rb.readBigWig(data)
        assert ei.value.code == _lib.RCP_ERR_DATA, name
    with pytest.raises(rb.RecoupError) as ei:
        rb.readBigWig(patched(kat_bytes(), 0, ">I", 0x888FFC26))
    assert ei.value.code == _lib.RCP_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_value_types_do_not_mix(bw_gpu):
    import ctypes as C
    rb = bw_gpu
    from recoup_b200 import _lib
    t = rb.readBigWig(kat_bytes())
    mask = rb.GRanges(np.zeros(2, np.int32), [1, 5], [10, 20], seqlevels=["chr1"])
    sig = rb.calcCoverage(t, mask)
    reads = rb.GRanges(np.zeros(3, np.int32), [1, 5, 9], [4, 8, 12], seqlevels=["chr1"], seqlengths=[1000])
    cnt = rb.calcCoverage(reads, mask)
    h = C.c_int(0)
    assert _lib.lib.rcp_coverage_concat3(sig.handle, cnt.handle, sig.handle, C.byref(h)) == _lib.RCP_ERR_ARG
    assert _lib.lib.rcp_coverage_concat3(sig.handle, sig.handle, sig.handle, C.byref(h)) == _lib.RCP_OK
    _lib.lib.rcp_coverage_free(h.value)
    buf = np.zeros(64, np.int32)
    ptr = np.zeros(3, np.int64)
    p64 = ptr.ctypes.data_as(C.POINTER(C.c_int64))
    i32 = buf.ctypes.data_as(C.POINTER(C.c_int32))
    assert _lib.lib.rcp_coverage_fetch(sig.handle, 0, 2, i32, 64) == _lib.RCP_ERR_ARG
    assert _lib.lib.rcp_coverage_rle(sig.handle, 0, 2, p64, None, None, 0) == _lib.RCP_ERR_ARG
    assert _lib.lib.rcp_coverage_fetch_f32(cnt.handle, 0, 2, buf.ctypes.data, 64) == _lib.RCP_ERR_ARG
    assert _lib.lib.rcp_coverage_rle_f32(cnt.handle, 0, 2, p64, None, None, 0) == _lib.RCP_ERR_ARG
    assert cnt.dtype == np.int32 and sig.dtype == np.float32
    assert sig[1].tolist() == [1.5] * 6 + [0.0] * 10
    t.free()


@pytest.mark.gpu
def test_bam_and_bigwig_samples_in_one_run(bw_gpu, tmp_path, fixture_data):
    """A BAM sample and a BigWig sample through coverageRef -> profileMatrix together."""
    rb = bw_gpu
    from tests.helpers import fixture_genes
    bam = rb.readBam(os.path.join(ROOT, "tests", "golden", "WT_H4K20me1_5kr.bam"))
    o_genes, genes = fixture_genes(fixture_data)
    size = int(bam.seqlengths[bam.seqlevels.index("chr12")])
    chroms = [("chr12", size)]
    rng = np.random.default_rng(9)
    lo, hi = int(o_genes["start"].min()) - 5000, int(o_genes["end"].max()) + 5000
    pos, items = max(lo, 0), []
    while pos < min(hi, size - 100):
        s = pos + int(rng.integers(0, 300))
        e = s + int(rng.integers(1, 200))
        items.append((s, e, float(np.float32(rng.gamma(2.0, 3.0)))))
        pos = e
    secs = [dict(chrom=0, type="bedGraph", items=items[i:i + 500]) for i in range(0, len(items), 500)]
    path = str(tmp_path / "signal.bw")
    with open(path, "wb") as f:
        f.write(write_bigwig(chroms, secs))
    genes = rb.GRanges(np.zeros(len(genes), np.int32), genes.start, genes.end, strand=genes.strand,
                       seqlevels=["chr12"], names=genes.names)
    inp = [dict(id="bam", name="bam", ranges=bam), dict(id="bw", name="bw", file=path, format="bigwig", ranges=None)]
    rb.coverageRef(inp, genes, "tss", (2000, 2000))
    bp = dict(flankBinSize=0, regionBinSize=100, sumStat="mean", interpolation="auto")
    rb.profileMatrix(inp, (2000, 2000), bp)
    solo = [dict(id="bam", name="bam", ranges=bam)]
    rb.coverageRef(solo, genes, "tss", (2000, 2000))
    rb.profileMatrix(solo, (2000, 2000), bp)
    assert np.array_equal(np.asarray(inp[0]["profile"]), np.asarray(solo[0]["profile"]))
    oracle = BO.Track.from_file_items(items_of(secs), [size])
    s, e = O.get_regional_ranges(o_genes["start"], o_genes["end"], o_genes["strand"], "tss", (2000, 2000))
    want_cov = BO.calc_coverage(oracle, dict(chrom=np.zeros(len(s), np.int64), start=s, end=e,
                                             strand=o_genes["strand"]))
    assert_signal_equal(inp[1]["coverage"].to_list(), want_cov)
    want = O.profile_matrix(want_cov, (2000, 2000), bp)
    absm = O.profile_matrix([None if c is None else np.abs(c) for c in want_cov], (2000, 2000), bp)
    assert_bins_close(inp[1]["profile"], want, absm)
