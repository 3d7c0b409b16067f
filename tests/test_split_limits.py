"""The split path at each of its geometries.

A candidate word of the split path holds P position bits (16 <= P <= 22, from the genome span
alone), 2 strand bits on stranded calls and the read width in what is left, capped at 8191.  The
cases put genomes on both sides of every P threshold and of the 32-bit coordinate limit, reads of
exactly the widest width a GRanges call packs and one base wider (the call must leave the split
path then, in eager mode before the plan and in deferred mode through its give_up() branch), the
handle's long-read list of the GRangesList path on both sides of its threshold and of its n / 8
rule, and reads across 2^P group, 16 kb bitmap-block and 1 kb sub-bin boundaries and chromosome
ends.  Coverage must equal the oracle bit for bit in eager and in deferred mode, and the fused
profile the two-stage one exactly.

Genomes reach 2^32 positions, but nothing is sized by the genome: reads sit in a few windows and
the oracle works region by region.  The CPU meta-test restates the geometry rules and fails when
the case table stops straddling a threshold.  Run the GPU tests with `-m gpu` on a B200."""
import ctypes as C

import numpy as np
import pytest

from oracle import recoup_oracle as O
from tests.helpers import assert_coverage_equal
from tests.test_deferred_validation import Sample, consume, list_mask, oracle_result, set_deferred, vp

SEED = 42

# ---- restated from the library ---------------------------------------------------------------
MIN_P, MAX_P, MAX_GROUPS = 16, 22, 1024      # rcp_internal.cuh:275-279 (split_position_bits)
WIDTH_CAP = 8191                             # coverage_split.cu:1676,1760
MAX_SPAN = 2**32 - 16                        # index.cu:590: a span from here on is RCP_ERR_UNSUPPORTED
PATH_SPLIT = 4


def position_bits(span):
    """split_position_bits: the fewest P >= 16 with ceil(span / 2^P) <= 1024, at most 22."""
    P = MIN_P
    while P < MAX_P and -(-span // (1 << P)) > MAX_GROUPS:
        P += 1
    return P


def width_limit(P, stranded):
    """The widest read a GRanges call packs (coverage_split.cu:1672-1676,1760: the call leaves the
    split path when max_w > 8191 or max_w >= 2^wbits)."""
    wbits = 32 - P - (2 if stranded else 0)
    return min((1 << wbits) - 1, WIDTH_CAP)


def long_thr(P, reads_have_strand):
    """index.cu:672-673: set at load from whether the READS have strands, not from the call."""
    wbits = 32 - P - (2 if reads_have_strand else 0)
    return min((1 << wbits) - 1, WIDTH_CAP) if wbits >= 7 else 0xffffffff


def long_list_serves(n, n_long):
    """coverage_split.cu:1605: more than n / 8 reads wider than the words: no binned index."""
    return n_long <= n // 8


# ---- the case table --------------------------------------------------------------------------
# spans on both sides of every P threshold (P = k up to 2^(k+10), k + 1 above it)
THRESHOLD_SPANS = [s for k in range(MIN_P, MAX_P) for s in (2**(k + 10), 2**(k + 10) + 1)]
# one genome per P for the width limits: the largest span of that P
P_SPANS = {P: (2**(P + 10) if P < MAX_P else MAX_SPAN - 1) for P in range(MIN_P, MAX_P + 1)}
UNSUPPORTED_SPANS = [MAX_SPAN - 1, MAX_SPAN]
WIDTH_CASES = [(P, stranded, side) for P in range(MIN_P, MAX_P + 1) for stranded in (False, True)
               for side in ("at", "past")]
N_LIST = 4000
LONG_CASES = [("at", 1), ("over", 0), ("over", 1)]     # (width vs long_thr, n_long - n // 8)
LONG_P = 22

A_LEN = 120_000                   # chromosome 0
B_LEN = (1 << MAX_P) + 6000       # chromosome 2: holds a 2^P group boundary for every P


def genome(span):
    """[A, filler, B, filler]: sum(len + 2) == span; every length fits a 32-bit read coordinate."""
    fill = span - (A_LEN + 2) - (B_LEN + 2) - 4
    f1 = fill // 2
    return [A_LEN, f1, B_LEN, fill - f1]


def offsets(clen):
    return np.concatenate([[0], np.cumsum(np.asarray(clen, np.int64) + 2)])


def special_points(clen, P):
    """(chrom, pos) where reads and windows go: a 2^P group boundary, a 16 kb block boundary and a
    1 kb sub-bin boundary on chromosome 2, a group boundary near the end of the last chromosome
    (global coordinates near the span), and the last base of chromosomes 0, 1 and 2."""
    off = offsets(clen)
    pts = []
    for c, lo in ((2, 1000), (2, 300_000), (2, 700_000)):
        for b in ((1 << P), 1 << 14, 1 << 10):
            g = -(-(off[c] + lo) // b) * b
            pts.append((c, int(g - off[c])))
    g3 = (off[3] + clen[3] - 20_000) // (1 << P) * (1 << P)
    pts.append((3, int(max(g3 - off[3], 30_000))))
    pts.append((3, int(clen[3] - 5000)))
    pts += [(0, clen[0]), (1, clen[1]), (2, clen[2])]
    return pts


def make_reads(rng, clen, P, widths=(), n_bg=2500, max_w=300):
    """Reads narrower than max_w on chromosome 0 and around the special points (some ending on a
    chromosome's last base), plus reads of each width in `widths` across every point."""
    cs, ss, es = [], [], []

    def add(c, s, e):
        s, e = max(int(s), 1), min(int(e), int(clen[c]))
        if s <= e:
            cs.append(c); ss.append(s); es.append(e)
    for _ in range(n_bg):
        w = int(rng.integers(1, max_w))
        s = int(rng.integers(1, clen[0] - w + 2))
        add(0, s, s + w - 1)
    for c, pos in special_points(clen, P):
        for _ in range(60):
            w = int(rng.integers(1, max_w))
            s = pos + int(rng.integers(-350, 350))
            add(c, s, s + w - 1)
        add(c, pos - 40, pos)                    # ends on the point (a chromosome's last base)
        for w in widths:
            for d in (-w // 2, -w + 1, 0, -w // 3):
                add(c, pos + d, pos + d + w - 1)
    n = len(cs)
    strand = rng.choice(np.array([1, -1, 0], np.int8), size=n)
    return np.asarray(cs, np.int32), np.asarray(ss, np.int64), np.asarray(es, np.int64), strand


def make_windows(rng, clen, P, lengths=(1, 50, 1024, 1025, 3000, 9000)):
    """Windows on every special point, and windows from position 1 of the chromosomes whose
    predecessor has reads on its last base."""
    c, s, L = [], [], []
    for ch, pos in special_points(clen, P):
        for ln in lengths:
            for d in (-ln // 2, -ln + 1, 0):
                c.append(ch); s.append(pos + d); L.append(ln)
    for ch in (1, 2, 3):
        for ln in (1, 500, 20_000):
            c.append(ch); s.append(1); L.append(ln)
    n = len(c)
    s = np.asarray(s, np.int64)
    return dict(chrom=np.asarray(c, np.int64), start=s, end=s + np.asarray(L, np.int64) - 1,
                strand=rng.choice(np.array([1, -1, 0]), size=n))


def equal_windows(rng, clen, P, L=3000):
    c, s = [], []
    for ch, pos in special_points(clen, P):
        for d in (-L // 2, -L + 1, 0, -7):
            c.append(ch); s.append(pos + d)
    s = np.asarray(s, np.int64)
    return dict(chrom=np.asarray(c, np.int64), start=s, end=s + L - 1,
                strand=rng.choice(np.array([1, -1, 0]), size=len(c)))


# ---- CPU meta-test ---------------------------------------------------------------------------
def test_case_table_straddles_every_threshold():
    # the closed form of the P rule: 16 up to 2^26, else k with 2^(k+9) < span <= 2^(k+10)
    rng = np.random.default_rng(0)
    for span in list(rng.integers(1, MAX_SPAN, size=2000)) + THRESHOLD_SPANS + [1, 2**26 - 1, MAX_SPAN - 1]:
        span = int(span)
        want = MIN_P if span <= 2**26 else next(k for k in range(MIN_P + 1, MAX_P + 1)
                                                 if 2**(k + 9) < span <= 2**(k + 10) or k == MAX_P)
        assert position_bits(span) == want, span
    # every threshold from 16 | 17 to 21 | 22, from both sides
    for k in range(MIN_P, MAX_P):
        below = [s for s in THRESHOLD_SPANS if position_bits(s) == k]
        above = [s for s in THRESHOLD_SPANS if position_bits(s) == k + 1]
        assert any(position_bits(s + 1) == k + 1 for s in below), k
        assert any(position_bits(s - 1) == k for s in above), k
    # the 32-bit limit, from both sides
    assert max(s for s in UNSUPPORTED_SPANS if s < MAX_SPAN) == MAX_SPAN - 1 and MAX_SPAN in UNSUPPORTED_SPANS
    # every genome the GPU tests build has the span it claims, 32-bit read coordinates and room
    # for the special points
    for span in THRESHOLD_SPANS + list(P_SPANS.values()) + UNSUPPORTED_SPANS:
        clen = genome(span)
        assert offsets(clen)[-1] == span and min(clen) >= 100_000 and max(clen) < 2**31 - 1
        P = position_bits(span)
        for c, pos in special_points(clen, P):
            assert 1 <= pos <= clen[c]
        assert any(c == 2 and (offsets(clen)[2] + pos) % (1 << P) == 0 for c, pos in special_points(clen, P))
    # one genome per P, each of that P; the widths cover limit and limit + 1 for both call kinds
    assert sorted(position_bits(s) for s in P_SPANS.values()) == list(range(MIN_P, MAX_P + 1))
    assert {(P, st) for P, st, side in WIDTH_CASES if side == "at"} == \
        {(P, st) for P, st, side in WIDTH_CASES if side == "past"} == \
        {(P, st) for P in range(MIN_P, MAX_P + 1) for st in (False, True)}
    limits = {(P, st): width_limit(P, st) for P in range(MIN_P, MAX_P + 1) for st in (False, True)}
    assert limits[(22, False)] == 1023 and limits[(22, True)] == 255 and limits[(16, True)] == 8191
    assert {limits[(P, False)] for P in range(MIN_P, 20)} == {WIDTH_CAP}      # the cap binds ...
    assert limits[(17, True)] == WIDTH_CAP and limits[(18, True)] == 4095     # ... and the word does
    # the long-read list: widths at and past long_thr, n_long at n/8 and n/8 + 1
    assert long_thr(LONG_P, True) == 255 and long_thr(LONG_P, False) == 1023
    for n in (N_LIST, N_LIST + 931, 8 * 1000 + 7):
        assert long_list_serves(n, n // 8) and not long_list_serves(n, n // 8 + 1)
    assert {extra for side, extra in LONG_CASES if side == "over"} == {0, 1}
    assert ("at", 1) in LONG_CASES        # n / 8 + 1 reads exactly long_thr wide: no long-read list needed


# ---- GPU -------------------------------------------------------------------------------------
MODES = ("eager", "deferred")


def _lib():
    from recoup_b200 import _lib as L
    return L


def _load(mode, chrom, s, e, st, clen):
    smp = Sample("dense", chrom, s, e, st, clen)
    set_deferred(mode == "deferred")
    try:
        return smp, smp.load()
    finally:
        set_deferred(0)


def _path_of(h_reads, mask, ignore, filt):
    """rcp_coverage + rcp_coverage_path_info: (coverage list, path)."""
    from recoup_b200.coverage import CoverageList
    L = _lib()
    c = np.ascontiguousarray(mask["chrom"], np.int32)
    s = np.ascontiguousarray(mask["start"], np.int32)
    e = np.ascontiguousarray(mask["end"], np.int32)
    st = np.ascontiguousarray(mask["strand"], np.int8)
    h = C.c_int(0)
    L.check(L.lib.rcp_coverage(h_reads, c.shape[0], vp(c), vp(s), vp(e), vp(st), ignore,
                               L.STRAND_ANY if filt is None else filt, L.MEM_HOST, C.byref(h)))
    pth, cand = C.c_int(0), C.c_int64(0)
    L.check(L.lib.rcp_coverage_path_info(h.value, C.byref(pth), C.byref(cand)))
    cov = CoverageList(h.value)
    got = cov.to_list()
    cov.free()
    return got, pth.value


def _fused_equals_two_stage(h_reads, mask, ignore, filt, n_bins=50):
    """rcp_coverage_profile against rcp_coverage + rcp_profile_matrix on the same handle: exact."""
    from recoup_b200.coverage import CoverageList
    L = _lib()
    c = np.ascontiguousarray(mask["chrom"], np.int32)
    s = np.ascontiguousarray(mask["start"], np.int32)
    e = np.ascontiguousarray(mask["end"], np.int32)
    st = np.ascontiguousarray(mask["strand"], np.int8)
    R = c.shape[0]
    filt = L.STRAND_ANY if filt is None else filt
    fused = np.full((n_bins, R), -7.0)
    nul = np.zeros(R, np.uint8)
    L.check(L.lib.rcp_coverage_profile(h_reads, R, vp(c), vp(s), vp(e), vp(st), ignore, filt, n_bins, SEED, 0,
                                       1.0, vp(fused), R, vp(nul), L.MEM_HOST))
    h = C.c_int(0)
    L.check(L.lib.rcp_coverage(h_reads, R, vp(c), vp(s), vp(e), vp(st), ignore, filt, L.MEM_HOST, C.byref(h)))
    two = np.full((n_bins, R), -9.0)
    rc = L.lib.rcp_profile_matrix(h.value, 1, 0, 0, 0, n_bins, 0, 0, SEED, 0, vp(two), R, L.MEM_HOST)
    cov = CoverageList(h.value)
    null = cov.is_null()
    cov.free()
    L.check(rc)
    assert np.array_equal(nul.astype(bool), null)
    assert np.array_equal(fused, two)
    return fused.T


def _is_split_tried(request):
    return request.node.callspec.params["gpu"] in ("auto", "split")


@pytest.mark.gpu
@pytest.mark.parametrize("span", THRESHOLD_SPANS)
def test_position_bit_thresholds(gpu, span):
    """Both sides of every P threshold: boundary reads and windows, both call kinds, both modes."""
    L = _lib()
    clen = genome(span)
    P = position_bits(span)
    rng = np.random.default_rng(span % 100_003)
    chrom, s, e, st = make_reads(rng, clen, P)
    o_reads = O.Reads(chrom, s, e, st, clen)
    mask = make_windows(rng, clen, P)
    eqm = equal_windows(rng, clen, P)
    bp = dict(flankBinSize=0, regionBinSize=50, sumStat="mean", interpolation="auto")
    for ignore, filt in ((1, None), (0, None), (1, -1)):
        want = O.calc_coverage(o_reads, mask, filt, bool(ignore))
        want_m = O.profile_matrix(O.calc_coverage(o_reads, eqm, filt, bool(ignore)), (0, 0), bp, seed=SEED)
        for mode in MODES:
            smp, h = _load(mode, chrom, s, e, st, clen)
            try:
                got, _ = _path_of(h, mask, ignore, filt)
                assert_coverage_equal(got, want)
                m = _fused_equals_two_stage(h, eqm, ignore, filt)
                np.testing.assert_allclose(m, want_m, rtol=1e-6, atol=1e-12)
            finally:
                L.lib.rcp_reads_free(h)


@pytest.mark.gpu
@pytest.mark.parametrize("P,stranded,side", WIDTH_CASES)
def test_read_width_limit(gpu, request, P, stranded, side):
    """Reads exactly as wide as the packed word allows stay on the split path; one base wider
    leaves it (eager: before the plan; deferred: give_up() after the plan fetch).  Coverage equals
    the oracle either way."""
    L = _lib()
    span = P_SPANS[P]
    clen = genome(span)
    assert position_bits(span) == P
    W = width_limit(P, stranded) + (side == "past")
    rng = np.random.default_rng(1000 * P + 2 * W + stranded)
    chrom, s, e, st = make_reads(rng, clen, P, widths=(W,), n_bg=1500, max_w=min(300, W))
    assert (e - s + 1).max() == W
    o_reads = O.Reads(chrom, s, e, st, clen)
    mask = make_windows(rng, clen, P, lengths=(1, 1025, W, 3 * W))
    ignore, filt = (0, None) if stranded else (1, None)
    want = O.calc_coverage(o_reads, mask, filt, bool(ignore))
    for mode in MODES:
        smp, h = _load(mode, chrom, s, e, st, clen)
        try:
            got, path = _path_of(h, mask, ignore, filt)
            assert_coverage_equal(got, want)
            if _is_split_tried(request):
                assert (path == PATH_SPLIT) == (side == "at"), (mode, path)
            _fused_equals_two_stage(h, equal_windows(rng, clen, P), ignore, filt)
        finally:
            L.lib.rcp_reads_free(h)
    # the other call kind on the same reads: stranded calls pack fewer width bits
    if stranded and side == "past" and W <= width_limit(P, False):
        smp, h = _load("deferred", chrom, s, e, st, clen)
        try:
            got, path = _path_of(h, mask, 1, None)
            assert_coverage_equal(got, O.calc_coverage(o_reads, mask, None, True))
            if _is_split_tried(request):
                assert path == PATH_SPLIT
        finally:
            L.lib.rcp_reads_free(h)


@pytest.mark.gpu
@pytest.mark.parametrize("na", [False, True])
@pytest.mark.parametrize("span", UNSUPPORTED_SPANS)
def test_genome_at_the_32_bit_limit(gpu, span, na):
    """span = 2^32 - 17 loads (P = 22); 2^32 - 16 is RCP_ERR_UNSUPPORTED, with known lengths and with
    NA lengths (whose stand-ins are the largest read end per chromosome), eager or deferred."""
    from recoup_b200 import RecoupError
    L = _lib()
    clen = genome(span)
    rng = np.random.default_rng(3)
    chrom, s, e, st = make_reads(rng, clen, MAX_P, n_bg=500)
    for c in range(4):                          # a read on the last base of every chromosome
        chrom = np.append(chrom, np.int32(c)); s = np.append(s, clen[c] - 9); e = np.append(e, clen[c])
        st = np.append(st, np.int8(1))
    load_len = np.full(4, -1, np.int64) if na else np.asarray(clen, np.int64)
    o_reads = O.Reads(chrom, s, e, st, load_len)
    mask = make_windows(rng, clen, MAX_P, lengths=(1, 3000))
    for mode in MODES:
        if span >= MAX_SPAN:
            with pytest.raises(RecoupError) as ei:
                _load(mode, chrom, s, e, st, load_len)
            assert ei.value.code == L.RCP_ERR_UNSUPPORTED
            continue
        smp, h = _load(mode, chrom, s, e, st, load_len)
        try:
            for ignore in (1, 0):
                got, _ = _path_of(h, mask, ignore, None)
                assert_coverage_equal(got, O.calc_coverage(o_reads, mask, None, bool(ignore)))
        finally:
            L.lib.rcp_reads_free(h)


@pytest.mark.gpu
@pytest.mark.parametrize("side,extra", LONG_CASES)
@pytest.mark.parametrize("has_strand", [True, False])
def test_long_read_list_of_the_binned_index(gpu, has_strand, side, extra):
    """GRangesList calls build the handle's binned index; reads wider than long_thr (set by whether
    the reads have strands) go to its long-read list while there are at most n / 8 of them, else the
    call takes the start-sorted pairs.  The GRanges calls that follow reuse what the list call built."""
    L = _lib()
    clen = genome(P_SPANS[LONG_P])
    thr = long_thr(LONG_P, has_strand)
    W = thr if side == "at" else thr + 1
    rng = np.random.default_rng(7 * extra + has_strand + (side == "at"))
    chrom, s, e, st = make_reads(rng, clen, LONG_P, n_bg=N_LIST, max_w=thr)
    n = chrom.shape[0]
    n_wide = n // 8 + extra
    pick = rng.choice(N_LIST, size=n_wide, replace=False)          # background reads on chromosome 0
    s[pick] = rng.integers(1, clen[0] - W + 2, size=n_wide)
    e[pick] = s[pick] + W - 1
    assert (e - s + 1).max() == W
    assert int(((e - s + 1) > thr).sum()) == (n_wide if side == "over" else 0)
    assert long_list_serves(n, n_wide) == (extra == 0)
    if not has_strand:
        st = None
    o_reads = O.Reads(chrom, s, e, np.zeros(n, np.int8) if st is None else st, clen)
    lm = list_mask(rng, o_reads, 150)
    mask = make_windows(rng, clen, LONG_P, lengths=(1, 1025, 3000))
    for mode in MODES:
        smp, h = _load(mode, chrom, s, e, st, clen)
        try:
            for cons in ("list", "cov_any", "cov_stranded", "cov_plus"):
                m = lm if cons == "list" else mask
                assert_coverage_equal(consume(h, cons, m)[1], oracle_result(cons, o_reads, m)[1])
        finally:
            L.lib.rcp_reads_free(h)
