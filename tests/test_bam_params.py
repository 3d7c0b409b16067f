"""ScanBamParam filters in the device BAM decoder (rcp_bam_decode_param): flag, mapqFilter,
simpleCigar, tagFilter and which, against the oracle's restatement of readGAlignments(file,
param = ...) (oracle/scanbam_oracle.py, items 1-6) on files the tests write themselves and on the
reference's own sample (tests/golden/WT_H4K20me1_5kr.bam).  Integer results: BIT-EXACT."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import import_oracle as IO
from oracle import recoup_oracle as O
from oracle import scanbam_oracle as SO
from recoup_b200.readers import ScanBamParam, scanBamFlag
from tests.bam_aux_writer import aux_field, bam_record
from tests.bam_writer import bam_file

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_BAM = os.path.join(HERE, "golden", "WT_H4K20me1_5kr.bam")
REFS = [("chr1", 50000), ("chr2", 30000), ("chrM", 900)]
CIGARS = ["36M", "10M500N26M", "5S20M3I11M", "12M2D8M1000N4M4D10M", "3H10=1X25=", "20M1P16M",
          "8M30N8M40N8M50N12M", "36S", "6I", "10M5N2I5N10M", "4D", "15M2000N", "7N20M", "10M5M", "40M"]


def _decode(raw, params, split=False):
    names, lens, first = IO.bam_header(raw)
    return SO.bam_decode(raw[first:], lens, split=split, params=params, seqnames=names)


def _cols(got):
    return got[0].tolist(), got[1].tolist(), got[2].tolist(), got[3].tolist()


# ------------------------------------------------------------------------------- CPU ------------
def test_scan_bam_flag_encodings():
    assert scanBamFlag() == (0xfff, 0xfff)
    assert scanBamFlag(isDuplicate=False) == (0xfff, 0xfff & ~0x400)
    assert scanBamFlag(isMinusStrand=True) == (0xfff & ~0x10, 0xfff)
    assert scanBamFlag(isPaired=True, isSupplementaryAlignment=False) == (0xffe, 0x7ff)
    # readGAlignments ANDs isUnmappedQuery = FALSE into whatever the user passes
    assert ScanBamParam().keep_words() == (0xfff, 0xffb)
    assert ScanBamParam(flag=scanBamFlag(isUnmappedQuery=True)).keep_words() == (0xffb, 0xffb)


def test_scan_bam_param_validation():
    for kw in (dict(tagFilter={"NHX": [1]}), dict(tagFilter={"N": [1]}), dict(tagFilter={"NH": [1, "a"]}),
               dict(tagFilter={"NH": [1.5]}), dict(mapqFilter=-1), dict(flag=(0x1fff, 0)),
               dict(which=[("chr1", 0, 10)]), dict(which=[("chr1", 10, 9)]), dict(which=[("chr1", 1, 536870913)]),
               dict(simpleCigar=1)):
        with pytest.raises(ValueError):
            ScanBamParam(**kw)
    with pytest.raises(ValueError):
        scanBamFlag(isDuplicate=1)
    p = ScanBamParam(which=[("chr2", 5, 9), ("chr1", 1, 3), ("chr2", 1, 2)], tagFilter={"NH": 1, "RG": ["a", "b"]},
                     what=["seq"], tag=["NM"], reverseComplement=True)
    assert p.which == [("chr2", 5, 9), ("chr2", 1, 2), ("chr1", 1, 3)]       # by level, given order within
    assert p.tagFilter == {"NH": [1], "RG": ["a", "b"]}


def test_oracle_without_params_is_the_plain_reader():
    rng = np.random.default_rng(3)
    raw, _ = _random_bam(rng, 600)
    names, lens, first = IO.bam_header(raw)
    for split in (False, True):
        for a, b in zip(SO.bam_decode(raw[first:], lens, split=split), IO.bam_decode(raw[first:], lens, split=split)):
            assert a.dtype == b.dtype and np.array_equal(a, b)


def test_oracle_each_filter_alone():
    recs = [bam_record(0, 99, 0, "36M", mapq=0), bam_record(0, 100, 1024, "36M", mapq=10),
            bam_record(0, 101, 16, "10M5M", mapq=255), bam_record(0, 102, 256 + 16, "36M", mapq=30),
            bam_record(0, 103, 4, "36M", mapq=60)]
    raw, _ = bam_file(REFS, recs)
    assert _cols(_decode(raw, None))[1] == [100, 101, 102, 103]
    assert _cols(_decode(raw, dict(flag=scanBamFlag(isDuplicate=False))))[1] == [100, 102, 103]
    assert _cols(_decode(raw, dict(flag=scanBamFlag(isMinusStrand=True))))[1] == [102, 103]
    assert _cols(_decode(raw, dict(flag=scanBamFlag(isSecondaryAlignment=False, isMinusStrand=True))))[1] == [102]
    assert _cols(_decode(raw, dict(flag=scanBamFlag(isUnmappedQuery=True))))[1] == []
    assert _cols(_decode(raw, dict(mapqFilter=10)))[1] == [101, 102, 103]      # 255 is the number 255
    assert _cols(_decode(raw, dict(mapqFilter=0)))[1] == [100, 101, 102, 103]
    assert _cols(_decode(raw, dict(simpleCigar=True)))[1] == [100, 101, 103]   # 10M5M is not simple


def test_oracle_tag_filter_walks_every_aux_type():
    before = (aux_field("XB", "B", [1.5, 2.5, -1.0], sub="f") + aux_field("MD", "Z", "10A25") +
              aux_field("XH", "H", "1AE3") + aux_field("XS", "B", [1, -2], sub="s") + aux_field("XF", "f", 0.5))
    recs = [bam_record(0, 10, 0, "36M", l_seq=5, tags=before + aux_field("NH", "C", 1)),
            bam_record(0, 11, 0, "36M", l_seq=4, tags=before + aux_field("NH", "i", 2)),
            bam_record(0, 12, 0, "36M", tags=aux_field("NM", "c", -1)),                   # NH missing
            bam_record(0, 13, 0, "36M", tags=aux_field("NH", "Z", "1")),                  # NH of the wrong type
            bam_record(0, 14, 0, "36M", tags=aux_field("NH", "f", 1.0)),                  # NH of the wrong type
            bam_record(0, 15, 0, "36M", tags=aux_field("NH", "s", 1) + aux_field("NH", "i", 2)),   # first wins
            bam_record(0, 16, 0, "36M", tags=aux_field("NH", "I", 1) + aux_field("RG", "A", "b")),
            bam_record(0, 17, 0, "36M", tags=aux_field("NH", "S", 1) + aux_field("RG", "Z", "grp"))]
    raw, _ = bam_file(REFS, recs)
    assert _cols(_decode(raw, dict(tagFilter={"NH": [1]})))[1] == [11, 16, 17, 18]
    assert _cols(_decode(raw, dict(tagFilter={"NH": [1, 2]})))[1] == [11, 12, 16, 17, 18]
    assert _cols(_decode(raw, dict(tagFilter={"NH": [1], "RG": ["b", "grp"]})))[1] == [17, 18]
    assert _cols(_decode(raw, dict(tagFilter={"MD": ["10A25"], "NH": [2]})))[1] == [12]
    assert _cols(_decode(raw, dict(tagFilter={"XF": [0]})))[1] == []                          # f never matches
    fields = SO.parse_aux(before + aux_field("NH", "C", 1))
    assert [(t, ty) for t, ty, _ in fields] == [("XB", "B"), ("MD", "Z"), ("XH", "H"), ("XS", "B"), ("XF", "f"),
                                                ("NH", "C")]
    bad = bam_record(0, 10, 0, "36M", tags=aux_field("XB", "B", [1, 2, 3], sub="i")[:-2])  # runs past the record
    raw, _ = bam_file(REFS, [bad])
    with pytest.raises(ValueError):
        _decode(raw, dict(tagFilter={"NH": [1]}))
    assert _cols(_decode(raw, None))[1] == [11]                     # without a tagFilter the aux is not read


def test_oracle_which_order_multiplicity_and_edges():
    recs = [bam_record(0, 99, 0, "10M"),                   # [100, 109]
            bam_record(0, 105, 16, "10M"),                 # [106, 115]
            bam_record(0, 199, 0, "6I"),                   # zero reference width: [200, 199], rlen 1
            bam_record(0, 300, 0, "10M20000N10M"),         # [301, 20320], a long spliced read
            bam_record(1, 49, 0, "10M"),                   # chr2 [50, 59]
            bam_record(-1, -1, 4, "*")]                    # unplaced, last
    raw, _ = bam_file(REFS, recs)
    # two overlapping ranges: the second read is returned twice, range by range
    c, s, e, st = _cols(_decode(raw, dict(which=[("chr1", 101, 106), ("chr1", 106, 108)])))
    assert list(zip(s, e)) == [(100, 109), (106, 115), (100, 109), (106, 115)]
    c, s, e, st = _cols(_decode(raw, dict(which=[("chr1", 109, 110)])))
    assert list(zip(s, e)) == [(100, 109), (106, 115)]
    # chr2 listed first, but the seqlevels say chr1 first
    p = dict(which=[("chr2", 1, 100), ("chr1", 1, 100)], which_levels=["chr1", "chr2"])
    assert _cols(_decode(raw, p))[0] == [0, 1]
    assert _cols(_decode(raw, dict(which=[("chr2", 1, 100), ("chr1", 1, 100)])))[0] == [1, 0]
    # the zero-width alignment occupies position 200 for the overlap test, not for its range
    assert _cols(_decode(raw, dict(which=[("chr1", 200, 200)])))[1:3] == ([200], [199])
    assert _cols(_decode(raw, dict(which=[("chr1", 201, 300)])))[1] == []
    assert _cols(_decode(raw, dict(which=[("chr1", 199, 199)])))[1] == []
    # a spliced read reaches a range 20 kb away; split cuts every appearance at N
    assert _cols(_decode(raw, dict(which=[("chr1", 20310, 20400)])))[1:3] == ([301], [20320])
    assert _cols(_decode(raw, dict(which=[("chr1", 20310, 20400)]), split=True))[1:3] == ([301, 20311], [310, 20320])
    # unsorted records
    raw, _ = bam_file(REFS, [bam_record(0, 500, 0, "10M"), bam_record(0, 400, 0, "10M")])
    with pytest.raises(ValueError):
        _decode(raw, dict(which=[("chr1", 1, 100)]))
    assert _cols(_decode(raw, dict(mapqFilter=1)))[1] == [501, 401]


# ------------------------------------------------------------------------------- GPU ------------
AUX_KINDS = [("NH", "C"), ("NH", "i"), ("NH", "s"), ("NM", "c"), ("XI", "I"), ("XU", "S"), ("MD", "Z"),
             ("RG", "A"), ("XF", "f"), ("XH", "H"), ("XB", "B")]


def _random_aux(rng):
    out = b""
    for _ in range(int(rng.integers(0, 5))):
        tag, ty = AUX_KINDS[int(rng.integers(0, len(AUX_KINDS)))]
        if ty in "cC":
            out += aux_field(tag, ty, int(rng.integers(0 if ty == "C" else -3, 4)))
        elif ty in "sS":
            out += aux_field(tag, ty, int(rng.integers(0 if ty == "S" else -3, 4)))
        elif ty in "iI":
            out += aux_field(tag, ty, int(rng.integers(0 if ty == "I" else -3, 4)))
        elif ty == "Z":
            out += aux_field(tag, ty, ["36", "10A25", ""][int(rng.integers(0, 3))])
        elif ty == "A":
            out += aux_field(tag, ty, "ab"[int(rng.integers(0, 2))])
        elif ty == "f":
            out += aux_field(tag, ty, 1.0)
        elif ty == "H":
            out += aux_field(tag, ty, "1AE3")
        else:
            sub = "cCsSiIf"[int(rng.integers(0, 7))]
            vals = [float(x) if sub == "f" else int(x) for x in rng.integers(0, 5, size=int(rng.integers(0, 6)))]
            out += aux_field(tag, ty, vals, sub=sub)
    return out


def _random_bam(rng, n, sorted_=False):
    rows = []
    for i in range(n):
        ref = int(rng.integers(0, len(REFS)))
        pos0 = int(rng.integers(0, REFS[ref][1] - 10))
        flag = int(rng.integers(0, 1 << 12))
        if i % 97 == 0:
            ref, pos0, flag = -1, -1, 4
        rows.append((ref, pos0, flag, CIGARS[int(rng.integers(0, len(CIGARS)))], int(rng.integers(0, 256)),
                     int(rng.integers(0, 40)), _random_aux(rng)))
    if sorted_:
        rows.sort(key=lambda x: (x[0] < 0, x[0], x[1]))
    recs = [bam_record(ref, pos0, flag, cig, name=b"q%d" % i, l_seq=l_seq, tags=aux, mapq=mapq)
            for i, (ref, pos0, flag, cig, mapq, l_seq, aux) in enumerate(rows)]
    return bam_file(REFS, recs)


def _random_params(rng, which=None):
    p = {}
    if rng.random() < 0.6:
        kw = {}
        for name in ("isPaired", "isProperPair", "isUnmappedQuery", "isMinusStrand", "isSecondaryAlignment",
                     "isNotPassingQualityControls", "isDuplicate", "isSupplementaryAlignment", "isFirstMateRead"):
            if rng.random() < 0.25:
                kw[name] = bool(rng.random() < 0.5)
        p["flag"] = scanBamFlag(**kw)
    if rng.random() < 0.5:
        p["mapqFilter"] = int(rng.integers(0, 256))
    if rng.random() < 0.2:
        p["simpleCigar"] = True
    if rng.random() < 0.5:
        tf = {}
        for tag, vals in (("NH", [1, 2]), ("NM", [-1, 0]), ("MD", ["36", ""]), ("RG", ["a"]), ("XF", [1])):
            if rng.random() < 0.4:
                tf[tag] = vals
        p["tagFilter"] = tf
    if which is not None:
        p["which"] = which
    return p


def _assert_same(got, want):
    for g, w, what in zip(got, want, ("chrom", "start", "end", "strand")):
        assert g.shape == w.shape, "%s: %s != %s" % (what, g.shape, w.shape)
        assert np.array_equal(g, w), what


@pytest.fixture(scope="module")
def rb():
    import recoup_b200 as rb
    rb.init(0)
    rb.set_coverage_path("auto")
    return rb


def _device_decode(raw, params, split):
    """rcp_bam_decode_param on records and offsets that live in device memory"""
    import torch
    from recoup_b200 import _lib
    from recoup_b200.readers import DecodedGRanges, bam_decode_param
    names, lens, first = IO.bam_header(raw)
    rec = np.frombuffer(raw, dtype=np.uint8, offset=first)
    off = IO.bam_record_offsets(raw[first:])
    d_rec = torch.from_numpy(rec.copy()).cuda()
    d_off = torch.from_numpy(off.copy()).cuda()
    h, n = C.c_int(0), C.c_int64(0)
    _lib.check(bam_decode_param(C.c_void_p(d_rec.data_ptr()), rec.shape[0], C.c_void_p(d_off.data_ptr()),
                                off.shape[0] - 1, names, lens, split, _lib.MEM_DEVICE, ScanBamParam(**params), h, n))
    torch.cuda.synchronize()
    return DecodedGRanges(h.value, n.value, names, lens)


def _got(g):
    return g.seqnames, g.start, g.end, g.strand


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 255, 5000])
@pytest.mark.parametrize("sa", ["keep", "split", "remove"])
def test_filters_match_the_oracle(rb, n, sa):
    rng = np.random.default_rng(1000 + n + 7 * len(sa))
    raw, bgzf = _random_bam(rng, n)
    split = sa == "split"
    for trial in range(4):
        params = _random_params(rng)
        want = _decode(raw, params, split=split)
        if sa == "remove":
            keep = O.splice_remove(want[1], want[2], 0.75)[0] if want[0].shape[0] else np.zeros(0, dtype=bool)
            want = tuple(x[keep] for x in want)
        got = rb.readBam(bgzf, sa=sa, params=ScanBamParam(**params))
        assert len(got) == want[0].shape[0], params
        _assert_same(_got(got), want)
        if sa != "remove":
            _assert_same(_got(_device_decode(raw, params, split)), want)


def _sorted_which(rng):
    which = [("chr2", 100, 5000), ("chr1", 1, 50000), ("chr1", 2000, 2100), ("chr1", 2050, 2300),
             ("chrM", 850, 900), ("chr1", 49990, 50000), ("chr2", 29000, 29000)]
    for _ in range(20):
        ref = int(rng.integers(0, len(REFS)))
        s = int(rng.integers(1, REFS[ref][1]))
        which.append((REFS[ref][0], s, s + int(rng.integers(0, 3000))))
    which.append(("chrM", 5000, 6000))                         # no hits: beyond the reference
    return which


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 255, 12000])
@pytest.mark.parametrize("sa", ["keep", "split"])
def test_which_matches_the_oracle(rb, n, sa):
    """overlapping ranges, ranges without hits, a whole-chromosome range whose run spans several
    chunks (2048 records each), ranges on every reference, listed out of level order"""
    rng = np.random.default_rng(2000 + n)
    raw, bgzf = _random_bam(rng, n, sorted_=True)
    split = sa == "split"
    which = _sorted_which(rng)
    for trial in range(3):
        params = _random_params(rng, which) if trial else dict(which=which)
        want = _decode(raw, params, split=split)
        got = rb.readBam(bgzf, sa=sa, params=ScanBamParam(**params))
        assert len(got) == want[0].shape[0]
        _assert_same(_got(got), want)
        _assert_same(_got(_device_decode(raw, params, split)), want)
        if trial == 0 and n == 12000:
            assert int((want[0] == 0).sum()) > 2048           # chr1 alone: more than one chunk


@pytest.mark.gpu
def test_which_needs_sorted_records_and_known_seqnames(rb):
    from recoup_b200 import _lib
    raw, bgzf = bam_file(REFS, [bam_record(0, 500, 0, "10M"), bam_record(0, 400, 0, "10M", mapq=0)])
    with pytest.raises(_lib.RecoupError) as ei:
        rb.readBam(bgzf, params=ScanBamParam(which=[("chr1", 1, 1000)]))
    assert ei.value.code == _lib.RCP_ERR_DATA
    assert rb.readBam(bgzf, params=ScanBamParam(mapqFilter=1)).start.tolist() == [501]
    assert rb.readBam(bgzf).start.tolist() == [501, 401]
    with pytest.raises(ValueError):
        rb.readBam(bgzf, params=ScanBamParam(which=[("chrX", 1, 10)]))
    # a malformed aux field is an error when a tagFilter reads it
    raw, bgzf = bam_file(REFS, [bam_record(0, 5, 0, "10M", tags=aux_field("MD", "Z", "10")[:-1])])
    with pytest.raises(_lib.RecoupError) as ei:
        rb.readBam(bgzf, params=ScanBamParam(tagFilter={"NH": 1}))
    assert ei.value.code == _lib.RCP_ERR_DATA
    assert len(rb.readBam(bgzf, params=ScanBamParam(mapqFilter=3))) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("sa", ["keep", "split"])
def test_all_na_param_equals_the_plain_decode(rb, sa):
    rng = np.random.default_rng(31)
    raw, bgzf = _random_bam(rng, 4000)
    plain = rb.readBam(bgzf, sa=sa)
    got = rb.readBam(bgzf, sa=sa, params=ScanBamParam())
    _assert_same(_got(got), _got(plain))


@pytest.mark.gpu
def test_golden_bam_filters_and_coverage(rb, fixture_data):
    from tests.helpers import assert_coverage_equal, fixture_genes
    data = open(GOLDEN_BAM, "rb").read()
    raw = IO.bgzf_inflate(data)
    names, lens, first = IO.bam_header(raw)
    assert len(rb.readBam(data, params=ScanBamParam(mapqFilter=30))) == 5000      # MAPQ 255 everywhere
    flags = []
    p = first
    while p < len(raw):
        bs = int.from_bytes(raw[p:p + 4], "little", signed=True)
        flags.append(int.from_bytes(raw[p + 18:p + 20], "little"))
        p += 4 + bs
    minus = rb.readBam(data, params=ScanBamParam(flag=scanBamFlag(isMinusStrand=True)))
    assert len(minus) == sum(1 for f in flags if f & 16) and set(minus.strand.tolist()) == {-1}
    s0 = int(IO.bam_decode(raw[first:], lens)[1][2000])
    spec = dict(which=[("chr12", s0, s0 + 200000)], flag=scanBamFlag(isMinusStrand=False))
    want = SO.bam_decode(raw[first:], lens, params=spec, seqnames=names)
    reads = rb.readBam(data, params=ScanBamParam(**spec))
    assert want[0].shape[0] > 0
    _assert_same(_got(reads), want)
    reads = rb.readBam(data, params=ScanBamParam(**spec))          # fresh: nothing fetched before coverage
    o_genes, g_genes = fixture_genes(fixture_data)
    inp = [dict(id="s", name="s", ranges=reads)]
    rb.coverageRef(inp, g_genes, "tss", (2000, 2000))
    o_reads = O.Reads(want[0], want[1].astype(np.int64), want[2].astype(np.int64), want[3], lens)
    assert_coverage_equal(inp[0]["coverage"].to_list(), O.coverage_ref(o_reads, o_genes, "tss", (2000, 2000)))


@pytest.mark.gpu
def test_preprocess_ranges_downsamples_the_filtered_reads(rb, tmp_path):
    rng = np.random.default_rng(77)
    files = []
    for k in range(2):
        recs = []
        for i in range(3000 + 700 * k):
            ref = int(rng.integers(0, 2))
            recs.append(bam_record(ref, int(rng.integers(0, REFS[ref][1] - 2200)), int(rng.choice([0, 16, 1024, 1040])),
                                   ["36M", "10M500N26M"][i % 2], mapq=int(rng.integers(0, 60)),
                                   tags=aux_field("NH", "C", int(rng.integers(1, 3)))))
        raw, bgzf = bam_file(REFS, recs)
        path = tmp_path / ("f%d.bam" % k)
        path.write_bytes(bgzf)
        files.append((str(path), raw))
    spec = dict(flag=scanBamFlag(isDuplicate=False), mapqFilter=10, tagFilter={"NH": [1]})
    inp = [dict(id="a", name="a", file=files[0][0], format="bam"), dict(id="b", name="b", file=files[1][0], format="bam")]
    rb.preprocessRanges(inp, dict(normalize="downsample", spliceAction="split", seed=42), bamParams=ScanBamParam(**spec))
    decoded = [_decode(raw, spec, split=True) for _, raw in files]
    sizes = [d[0].shape[0] for d in decoded]
    assert sizes[0] != sizes[1] and max(sizes) < 3000
    assert len(inp[0]["ranges"]) == len(inp[1]["ranges"]) == min(sizes)
    idx = O.downsample_indices(sizes, "downsample", seed=42)
    for x, d, ix in zip(inp, decoded, idx):
        _assert_same(_got(x["ranges"]), tuple(a[ix - 1] for a in d))


@pytest.mark.gpu
def test_a_filter_that_removes_everything(rb):
    recs = [bam_record(0, 5, 0, "10M"), bam_record(1, 7, 16, "4M")]
    _, bgzf = bam_file(REFS, recs)
    for params in (ScanBamParam(mapqFilter=200), ScanBamParam(which=[("chrM", 1, 900)]),
                   ScanBamParam(tagFilter={"NH": [1]})):
        reads = rb.readBam(bgzf, params=params)
        assert len(reads) == 0 and reads.start.shape == (0,)
        mask = rb.GRanges(np.zeros(1, dtype=np.int32), [1], [100], strand=np.zeros(1, dtype=np.int8),
                          seqlevels=[r[0] for r in REFS])
        empty = rb.readBam(bam_file(REFS, [])[1])          # what the decoder already gives for no reads
        assert [np.asarray(x).tolist() if x is not None else None for x in rb.calcCoverage(reads, mask).to_list()] == \
               [np.asarray(x).tolist() if x is not None else None for x in rb.calcCoverage(empty, mask).to_list()]
