"""Every branch of the profile kernels against an exact reference, under each coverage storage:
uint16 counts (split path), int32 counts (RCP_COVERAGE_WIDE=1) and float32 signal (bigWig).

The coverage of each case is built from a target vector -- reads by level decomposition, or one
bedGraph item per run of equal values -- and fetched back bit for bit before anything is binned.
Values are adversarial: interior bases carry a hash of their position (0..7), the first and last
base of every bin 8..15, so a base counted in the wrong bin changes an integer sum.

Reference (plain numpy on the fetched coverage; only the bin layout comes from the oracle):
  * integer mean  scale * (float(int64 sum) / count), bit for bit;
  * median        scale * ((a + b) * 0.5) of the two middle values, bit for bit;
  * per base      scale * value, bit for bit;
  * float mean    math.fsum, within (count + 2) * 2^-53 * sum|x| * |scale| / count;
  * segments shorter than the bin count (interpolation): O.split_vector within 1e-11 of max|y|
    (the device contracts FMAs in the spline, so those rows are not bit-identical).

The branch meta-test restates the dispatch of bin_desc_kernel and the host sizing of
bin_matrix_impl (recoup_b200/csrc/profile.cu) and checks that the case matrix reaches every
branch under every storage.  Run the GPU tests with `-m gpu` on a B200."""
import ctypes as C
import math
import struct
from collections import namedtuple

import numpy as np
import pytest

from oracle import recoup_oracle as O
from tests.bigwig_writer import write_bigwig

STORAGES = ["narrow", "wide", "float32"]
SEED = 42

# ---- restated from recoup_b200/csrc/profile.cu ------------------------------------------------
STAGE_INTS = 12288            # ints of one staging buffer (48 KB)
STAGE_MAX_BIN = 128           # narrower bins are summed from shared memory
LONG_REGION_MIN = 16384       # wide bins of segments from this length on: bin_wide_kernel
NBUF_MAX = 8
WIDE_RUN = 16                 # bins of one bin_wide_kernel unit
CTAS_WIDE_BUF = 6144          # staging ints in the 8-CTAs-per-SM mode
MAX_BINS = 38399              # (n + 1 + 3) & ~3 ints of bin edges <= 150 KB
RRNG_BYTES = 624 * 4 + 8
INTERP_MAX_BINS = (220 * 1024 - 8 - RRNG_BYTES) // (4 * 8 + 2 * 4)      # 5569
FUSED_MAX_BINS = 30000        # coverage_split.cu: coverage_profile_split
BASE_WIDE_COLS = 128          # base_matrix_wide_kernel from this many columns on
BASE_SLAB_ROWS = 65535 * 32   # rows of one base_matrix_kernel launch (grid.y <= 65535)
FUSED_SMALL = 1 << 22         # a fused tile with coverage this high sums base by base
assert INTERP_MAX_BINS == 5569


def edge_bytes(n):
    return ((n + 1 + 3) & ~3) * 4


def segment(L, where, f1, f2):
    """segment_of(): [a, b) of a window of length L."""
    a, b = {"center": (f1, L - f2), "upstream": (0, f1), "downstream": (L - f2, L)}.get(where, (0, L))
    a = max(a, 0)
    b = max(min(b, L), a)
    return a, b


def auto_neighborhood(Ls, n):
    return (n - Ls) / n < 0.2                   # util.R:21 (same double expression as the kernel)


def host_plan(lens, n, where, f1, f2, ctas=None):
    """bin_matrix_impl (mean): staging ints per buffer, CTAs per SM, buffers per CTA."""
    live = [L for L in lens if L is not None]
    seg_max = max(live, default=0)
    seg_mean = sum(live) // max(len(live), 1)
    if where == "upstream":
        seg_max, seg_mean = min(seg_max, f1), min(seg_mean, f1)
    elif where == "downstream":
        seg_max, seg_mean = min(seg_max, f2), min(seg_mean, f2)
    elif where == "center":
        seg_max, seg_mean = max(seg_max - f1 - f2, 0), max(seg_mean - f1 - f2, 0)
    buf = min(STAGE_INTS, (seg_max + 18) & ~3)
    per_sm, mode8 = 4, False
    if seg_mean // n >= 128:
        per_sm, mode8, buf = 8, True, min(buf, CTAS_WIDE_BUF)
    if ctas is not None:
        per_sm = max(1, ctas)

    def budget(k):
        return 220 * 1024 // k - 1024
    while per_sm > 1 and budget(per_sm) - edge_bytes(n) < buf * 4:
        per_sm -= 1
    nbuf = min((budget(per_sm) - edge_bytes(n)) // (buf * 4), NBUF_MAX)
    assert nbuf >= 1
    return buf, per_sm, nbuf, mode8


def dispatch(L, n, where, f1, f2, buf, narrow):
    """bin_desc_kernel / bin_mean_kernel: the branch one window takes."""
    a, b = segment(L, where, f1, f2)
    Ls = b - a
    if Ls <= 0:
        return "empty"
    if Ls < n:
        return "neighborhood" if auto_neighborhood(Ls, n) else "spline"
    bsz = Ls // n
    sh = 3 if narrow else 2
    cap = ((buf >> 1) & ~3) if narrow else buf
    lo_al = a & ~((1 << sh) - 1)
    nvec = (b - lo_al + (1 << sh) - 1) >> sh
    if bsz < STAGE_MAX_BIN:
        return "staged" if nvec * 4 <= cap else "chunked"
    return "bin_wide" if Ls >= LONG_REGION_MIN else "cta_wide"


def median_group(bsz):
    g = 1
    while g < 32 and g < bsz:
        g <<= 1
    return g


# ---- the case matrix -------------------------------------------------------------------------
Case = namedtuple("Case", "n where f1 f2 scale kind R cap lens")


def ls_candidates(n, cap):
    c = []
    if n <= INTERP_MAX_BINS:                    # larger bin counts: short segments are the limits test
        if n >= 2:
            c.append(max(1, n // 2))            # spline
        if n >= 6:
            lo = next(Ls for Ls in range(4, n) if auto_neighborhood(Ls, n))
            c += [lo, lo - 1]                   # both sides of the auto threshold
    for w in (1, 2, 3, 5, 9, 17, 33, 127, 128, 200):
        c.append(w * n)                         # dif == 0
        if n > 1:
            c.append(w * n + max(1, n // 3))    # dif > 0
    c.append(STAGE_INTS + 107)                  # longer than any staging buffer
    c.append(max(LONG_REGION_MIN, 128 * n) + n // 2 + 5)
    return sorted(set(x for x in c if 1 <= x <= cap and (x >= n or n <= INTERP_MAX_BINS)))


def window_lengths(n, where, f1, f2, R, cap, ls_list=None, budget=250_000):
    """Window lengths (None: NULL) in one rotation over the region kinds, heavy kinds capped
    by a budget of bases each."""
    kinds = ["null"] + (["empty"] if where == "center" and f1 + f2 >= 3 else [])
    for Ls in ls_list if ls_list is not None else ls_candidates(n, cap):
        if where == "upstream" and Ls > f1 or where == "downstream" and Ls > f2:
            continue
        kinds.append(Ls)
    left = {k: (10 ** 9 if isinstance(k, str) or k <= 2000 else max(2, budget // k)) for k in kinds}
    out, i = [], 0
    while len(out) < R:
        progressed = False
        for k in kinds:
            if len(out) >= R or left[k] == 0:
                continue
            left[k] -= 1
            progressed = True
            i += 1
            if k == "null":
                out.append(None)
            elif k == "empty":
                out.append(max(1, f1 + f2 - i % 3))
            elif where == "whole":
                out.append(k)
            elif where == "center":
                out.append(k + f1 + f2)
            else:                               # a flank segment: longer windows end at the flank
                flank = f1 if where == "upstream" else f2
                out.append(k + (i % 7 if k == flank else 0))
        assert progressed
    return out


def make_case(n, where, f1, f2, scale, kind, R=2400, cap=45_000, ls_list=None, budget=250_000):
    return Case(n, where, f1, f2, scale, kind, R, cap,
                tuple(window_lengths(n, where, f1, f2, R, cap, ls_list, budget)))


BIN_CASES = [
    make_case(1, "whole", 0, 0, 1.0, "Rejection"),
    make_case(3, "center", 3, 300, 0.37, "Rounding"),
    make_case(37, "center", 1001, 3, 1.0, "Rejection"),
    make_case(37, "upstream", 1001, 300, 0.37, "Rejection"),
    make_case(37, "downstream", 0, 1001, 1.0, "Rounding"),
    make_case(255, "whole", 0, 0, 0.37, "Rejection"),
    make_case(256, "center", 300, 300, 1.0, "Rejection"),
    make_case(257, "center", 3, 0, 1.0, "Rounding"),
    make_case(1024, "whole", 0, 0, 0.37, "Rejection", cap=135_000),
    make_case(6000, "whole", 0, 0, 1.0, "Rejection", R=300),
    make_case(MAX_BINS, "whole", 0, 0, 0.37, "Rounding", R=48, cap=80_000),
    # mostly wide bins: 8 CTAs per SM, 6 144-int buffers, chunked segments longer than those
    make_case(64, "whole", 0, 0, 1.0, "Rejection", R=400,
              ls_list=[30, 60, 5000, 8000, 12000, 16000, 20000], budget=10 ** 9),
]
KNOB = [None, 1, 2, 8, 16]                      # RCP_BIN_CTAS


def case_id(c):
    return "n%d-%s-%d-%d" % (c.n, c.where, c.f1, c.f2)


def branches_of(case, storage):
    """Every branch the case reaches under one storage (mean over the knob sweep, and median)."""
    narrow = storage == "narrow"
    hit = set()
    for ctas in KNOB:
        buf, per_sm, nbuf, mode8 = host_plan(case.lens, case.n, case.where, case.f1, case.f2, ctas)
        kernel_nbuf = min(2 * nbuf, NBUF_MAX) if narrow else nbuf
        if nbuf == 1:
            hit.add("nbuf1")                    # (narrow storage splits it into a ring of two)
        if kernel_nbuf > 1:
            hit.add("ring")
        if mode8:
            hit.add("per_sm8")
        for L in case.lens:
            if L is None:
                hit.add("null")
                continue
            b = dispatch(L, case.n, case.where, case.f1, case.f2, buf, narrow)
            hit.add(b)
            a, e = segment(L, case.where, case.f1, case.f2)
            Ls = e - a
            if b in ("staged", "chunked", "cta_wide", "bin_wide"):
                dif = Ls % case.n
                hit.add(b + ("_dif" if dif else "_equal"))
                if b == "bin_wide" and dif and case.n > WIDE_RUN:
                    hit.add("bin_wide_dif_runs")
                if b == "chunked" and mode8:
                    hit.add("chunked_per_sm8")
                if b == "staged" and nbuf == 1:
                    hit.add("staged_nbuf1")
                if b == "staged" and kernel_nbuf > 1:
                    hit.add("staged_ring")
                hit.add("median_g%d" % median_group(Ls // case.n))
            if a % 4:
                hit.add("unaligned_start")
            assert b in ("empty", "staged", "chunked", "cta_wide", "bin_wide") or case.n <= INTERP_MAX_BINS
    if case.n > INTERP_MAX_BINS:
        hit.add("many_bins")
    return hit


REQUIRED = {"null", "empty", "spline", "neighborhood", "staged", "chunked", "cta_wide", "bin_wide",
            "staged_equal", "staged_dif", "chunked_equal", "chunked_dif", "cta_wide_equal", "cta_wide_dif",
            "bin_wide_equal", "bin_wide_dif", "bin_wide_dif_runs", "per_sm8", "chunked_per_sm8", "nbuf1",
            "ring", "staged_nbuf1", "staged_ring", "unaligned_start", "many_bins"} | \
           {"median_g%d" % g for g in (1, 2, 4, 8, 16, 32)}


@pytest.mark.parametrize("storage", STORAGES)
def test_case_matrix_reaches_every_branch(storage):
    hit = set()
    for c in BIN_CASES:
        hit |= branches_of(c, storage)
        assert c.n <= MAX_BINS and edge_bytes(c.n) <= 150 * 1024
        assert len(c.lens) >= (2400 if c.n <= 1024 and c.n != 64 else 48)
        assert sum(L for L in c.lens if L) < 6_000_000
    assert REQUIRED <= hit, sorted(REQUIRED - hit)
    assert edge_bytes(MAX_BINS + 1) > 150 * 1024


# ---- targets and the coverages built from them --------------------------------------------------
INT_EDGE, INT_PILE = 8, 70_000
F_INTERIOR = np.array([0.0, -0.0, 1.0, -2.5, 0.1, 1e-40, 3.75, -7.0], dtype=np.float32)
F_EDGE = np.array([1e30, -1e30, 12.5, -0.3, 1e-38, 1e20, -3e10, 65536.5], dtype=np.float32)
GAP = 5


def hash8(pos):
    x = (np.asarray(pos, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)
    return (x & np.uint64(7)).astype(np.int64)


_layouts = {}


def layout(Ls, n, kind):
    """bin sizes (util.R:74-80); they depend on n and Ls % n only"""
    key = (n, Ls % n, kind)
    if key not in _layouts:
        _layouts[key] = O.bin_layout(n + Ls % n, n, SEED, kind) - 1
    return _layouts[key] + Ls // n


def targets_for(lens, n, where, f1, f2, kind, storage):
    """Start (1-based, chromosome c0) and target vector of every window; None for NULL."""
    starts, targets, pos = [], [], 1
    flt = storage == "float32"
    for i, L in enumerate(lens):
        if L is None:
            starts.append(None)
            targets.append(None)
            continue
        p = pos + np.arange(L)
        code = hash8(p)
        edge = np.zeros(L, dtype=bool)
        a, b = segment(L, where, f1, f2)
        if b - a >= n:
            fac = layout(b - a, n, kind)
            first = a + np.concatenate([[0], np.cumsum(fac)[:-1]])
            edge[first] = True
            edge[first + fac - 1] = True
        if flt:
            t = np.where(edge, F_EDGE[code], F_INTERIOR[code]).astype(np.float32)
        else:
            t = code + INT_EDGE * edge
            t[-1] += not t.any()                # zero reads would make the window NULL
            if storage == "wide" and i % 97 == 5 and b - a >= 4:
                t[a + 1:a + 4] += INT_PILE      # counts above 65 535: the int32 instances
        starts.append(pos)
        targets.append(t)
        pos += L + GAP
    return starts, targets, pos


def level_reads(G):
    """Reads (0-based inclusive) whose coverage is G: one read per maximal run of c >= h, for
    every level h, cut into pieces of at most 500 bases."""
    p = np.concatenate([[0], G, [0]]).astype(np.int64)
    d = np.diff(p)

    def expand(at, lo, cnt):
        tot = int(cnt.sum())
        k = np.arange(tot) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        return np.repeat(at, cnt), np.repeat(lo, cnt) + k
    up, dn = np.flatnonzero(d > 0), np.flatnonzero(d < 0)
    s_pos, s_lvl = expand(up, p[up] + 1, d[up])
    e_pos, e_lvl = expand(dn - 1, p[dn + 1] + 1, -d[dn])
    s = s_pos[np.lexsort((s_pos, s_lvl))]
    e = e_pos[np.lexsort((e_pos, e_lvl))]
    w = e - s + 1
    k = (w + 499) // 500
    ss = np.repeat(s, k) + 500 * (np.arange(int(k.sum())) - np.repeat(np.cumsum(k) - k, k))
    ee = np.minimum(ss + 499, np.repeat(e, k))
    return ss, ee


def genome_vector(starts, targets, clen, dtype):
    G = np.zeros(clen, dtype=dtype)
    for s, t in zip(starts, targets):
        if t is not None:
            G[s - 1:s - 1 + t.shape[0]] = t
    return G


def bedgraph_bigwig(starts, targets, clen):
    """One bedGraph item per run of equal values inside the windows; sections of 1 024 items."""
    s0, e0, v = [], [], []
    for s, t in zip(starts, targets):
        if t is None:
            continue
        bits = t.view(np.uint32)
        brk = np.flatnonzero(np.diff(bits) != 0) + 1
        a = np.concatenate([[0], brk])
        b = np.concatenate([brk, [t.shape[0]]])
        s0.append(s - 1 + a)
        e0.append(s - 1 + b)
        v.append(t[a])
    s0, e0, v = np.concatenate(s0), np.concatenate(e0), np.concatenate(v)
    secs = []
    for k in range(0, s0.shape[0], 1024):
        body = np.empty(min(1024, s0.shape[0] - k), dtype=[("s", "<u4"), ("e", "<u4"), ("v", "<f4")])
        body["s"], body["e"], body["v"] = s0[k:k + 1024], e0[k:k + 1024], v[k:k + 1024]
        lo, hi = int(body["s"][0]), int(body["e"][-1])
        head = struct.pack("<IIIIIBBH", 0, lo, hi, 0, 0, 1, 0, body.shape[0])
        secs.append({"raw": head + body.tobytes(), "box": (0, lo, 0, hi)})
    return write_bigwig([("c0", clen)], secs, compress=False)


def mask_arrays(starts, lens):
    chrom = np.array([1 if s is None else 0 for s in starts], dtype=np.int32)
    st = np.array([1 if s is None else s for s in starts], dtype=np.int64)
    ln = np.array([10 if L is None else L for L in lens], dtype=np.int64)
    return chrom, st, st + ln - 1


def normalised(t):
    """A target as the coverage holds it: -0.0 reads as +0.0."""
    return t if t.dtype != np.float32 else np.where(t == 0, np.float32(0), t).astype(np.float32)


def assert_same_coverage(got, targets):
    assert len(got) == len(targets)
    for r, (g, t) in enumerate(zip(got, targets)):
        if t is None:
            assert g is None, r
            continue
        assert g is not None and g.shape == t.shape, r
        t = normalised(t)
        if t.dtype == np.float32:
            assert np.array_equal(g.view(np.uint32), t.view(np.uint32)), r
        else:
            assert np.array_equal(g.astype(np.int64), t), r


class Store:
    """Coverage from target vectors under one storage type."""

    def __init__(self, name, rb, monkeypatch):
        self.name, self.rb, self.mp = name, rb, monkeypatch

    def storage_bytes(self, cov):
        from recoup_b200 import _lib
        b = C.c_int(0)
        _lib.check(_lib.lib.rcp_coverage_storage_bytes(cov.handle, C.byref(b)))
        return b.value

    def coverage(self, lens, starts, targets, clen, check=True):
        rb = self.rb
        chrom, ms, me = mask_arrays(starts, lens)
        mask = rb.GRanges(chrom, ms, me, strand=np.ones(len(lens), dtype=np.int8), seqlevels=["c0", "c1"])
        if self.name == "float32":
            track = rb.readBigWig(bedgraph_bigwig(starts, targets, clen))
            cov = rb.calcCoverage(track, mask)
            track.free()
        else:
            G = genome_vector(starts, targets, clen, np.int64)
            s, e = level_reads(G)
            reads = rb.GRanges(np.zeros(s.shape[0], dtype=np.int32), s + 1, e + 1,
                               strand=np.zeros(s.shape[0], dtype=np.int8), seqlevels=["c0", "c1"],
                               seqlengths=[clen, 1000])
            if self.name == "wide":
                self.mp.setenv("RCP_COVERAGE_WIDE", "1")
            else:
                self.mp.delenv("RCP_COVERAGE_WIDE", raising=False)
            cov = rb.calcCoverage(reads, mask)
            self.mp.delenv("RCP_COVERAGE_WIDE", raising=False)
            assert self.storage_bytes(cov) == (4 if self.name == "wide" else 2)
        if check:
            assert_same_coverage(cov.to_list(), targets)
        return cov


@pytest.fixture
def rb():
    import recoup_b200 as rb
    rb.init(0)
    rb.set_coverage_path("split")
    yield rb
    rb.set_coverage_path("auto")


@pytest.fixture(params=STORAGES)
def store(request, rb, monkeypatch):
    return Store(request.param, rb, monkeypatch)


# ---- the exact reference ------------------------------------------------------------------------
def reference(cov_list, n, where, f1, f2, scale, kind, stat):
    """(ref, tol): tol == 0 means bit for bit."""
    R = len(cov_list)
    ref = np.zeros((R, n))
    tol = np.zeros((R, n))
    for r, c in enumerate(cov_list):
        if c is None:
            continue
        a, b = segment(c.shape[0], where, f1, f2)
        x = c[a:b]
        Ls = b - a
        if Ls == 0:                 # empty segment (center window shorter than its flanks): zero row
            continue
        xd = x.astype(np.float64)
        if Ls < n:
            ref[r] = scale * O.split_vector(xd, n, "auto", "mean", SEED, kind)
            tol[r] = 1e-11 * np.abs(xd).max() * abs(scale)
            continue
        fac = layout(Ls, n, kind)
        st = np.concatenate([[0], np.cumsum(fac)[:-1]])
        if stat == "median":
            o = np.lexsort((xd, np.repeat(np.arange(n), fac)))
            xs = xd[o]
            ref[r] = scale * ((xs[st + (fac - 1) // 2] + xs[st + fac // 2]) * 0.5)
        elif x.dtype != np.float32:
            s = np.add.reduceat(x.astype(np.int64), st)
            ref[r] = scale * (s.astype(np.float64) / fac.astype(np.float64))
        else:
            xl = xd.tolist()
            sums = [math.fsum(xl[i:i + k]) for i, k in zip(st.tolist(), fac.tolist())]
            ref[r] = scale * (np.array(sums) / fac)
            tol[r] = (fac + 2) * 2.0 ** -53 * np.add.reduceat(np.abs(xd), st) * abs(scale) / fac
    return ref, tol


def assert_matches(got, ref, tol, what):
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == ref.shape, what
    exact = tol == 0
    bad = exact & (got.view(np.uint64) != ref.view(np.uint64))
    bad |= ~exact & ~(np.abs(got - ref) <= tol)
    if bad.any():
        r, c = np.argwhere(bad)[0]
        raise AssertionError("%s: %d entries differ; first [%d, %d]: got %r want %r (tol %g)"
                             % (what, int(bad.sum()), r, c, got[r, c], ref[r, c], tol[r, c]))


# ---- CPU checks of the builders and the reference -----------------------------------------------
def test_level_reads_give_the_target_coverage():
    lens = [None, 40, 7, 1, 300, None, 64]
    starts, targets, clen = targets_for(lens, 5, "whole", 0, 0, "Rejection", "narrow")
    targets[4][100:103] += 9000                     # a pile
    targets[1][:] = 0                               # all zero (a window without reads: NULL)
    G = genome_vector(starts, targets, clen, np.int64)
    s, e = level_reads(G)
    assert (e - s + 1).max() <= 500
    reads = O.Reads(np.zeros(s.shape[0]), s + 1, e + 1, np.zeros(s.shape[0]), [clen, 1000])
    chrom, ms, me = mask_arrays(starts, lens)
    got = O.calc_coverage(reads, dict(chrom=chrom, start=ms, end=me, strand=np.ones(len(lens))))
    want = [None if (t is None or not t.any()) else t for t in targets]
    assert_same_coverage(got, want)
    # the number of reads is the sum of the positive steps
    assert s.shape[0] >= int(np.maximum(np.diff(np.concatenate([[0], G])), 0).sum())


def test_bedgraph_items_give_the_target_signal():
    from oracle import bigwig_oracle as BO
    lens = [33, None, 5, 120]
    starts, targets, clen = targets_for(lens, 4, "whole", 0, 0, "Rounding", "float32")
    data = bedgraph_bigwig(starts, targets, clen)
    assert len(data) > 64
    items = []
    for s, t in zip(starts, targets):
        if t is not None:
            items += [(0, s - 1 + i, s + i, float(v)) for i, v in enumerate(t)]
    track = BO.Track.from_file_items(items, [clen])
    chrom, ms, me = mask_arrays(starts, lens)
    chrom = np.where(chrom == 1, -1, chrom)
    got = BO.calc_coverage(track, dict(chrom=chrom, start=ms, end=me, strand=np.ones(len(lens))))
    assert_same_coverage(got, targets)


@pytest.mark.parametrize("kind", ["Rejection", "Rounding"])
def test_reference_equals_split_vector(kind):
    """Integer means, medians and interpolated rows equal the oracle's splitVector bit for bit."""
    for n, where, f1, f2 in [(37, "center", 1001, 3), (5, "upstream", 300, 0), (256, "whole", 0, 0)]:
        lens = window_lengths(n, where, f1, f2, 60, 40_000)
        starts, targets, _ = targets_for(lens, n, where, f1, f2, kind, "narrow")
        for stat in ("mean", "median"):
            ref, tol = reference(targets, n, where, f1, f2, 1.0, kind, stat)
            for r, (L, t) in enumerate(zip(lens, targets)):
                if t is None:
                    assert not ref[r].any()
                    continue
                a, b = segment(L, where, f1, f2)
                if b == a:                      # empty segment: the oracle has no answer, the kernel a zero row
                    assert not ref[r].any()
                    continue
                want = O.split_vector(t[a:b], n, "auto", stat, SEED, kind)
                assert np.array_equal(ref[r], want), (n, where, r, stat)


def test_reference_float_mean_bound():
    x = np.array([1e30, 1.0, -1e30, 1e-40, 3.75], dtype=np.float32)
    ref, tol = reference([x], 1, "whole", 0, 0, 0.37, "Rejection", "mean")
    assert ref[0, 0] == 0.37 * (math.fsum(x.astype(np.float64).tolist()) / 5)
    assert 0 < tol[0, 0] < 1e15
    ref, tol = reference([np.zeros(4, dtype=np.float32)], 2, "whole", 0, 0, 1.0, "Rejection", "mean")
    assert not ref.any() and not tol.any()


# ---- GPU: bin matrices --------------------------------------------------------------------------
def bin_matrix(rb, cov, case, stat):
    flank = None if case.where == "whole" else (case.f1, case.f2)
    return np.asarray(rb.binCoverageMatrix(cov, binSize=case.n, stat=stat, flank=flank, where=case.where,
                                           sample_kind=case.kind))


@pytest.mark.gpu
@pytest.mark.parametrize("case", BIN_CASES, ids=case_id)
def test_bin_matrix_exact(store, case, monkeypatch):
    rb = store.rb
    starts, targets, clen = targets_for(case.lens, case.n, case.where, case.f1, case.f2, case.kind, store.name)
    cov = store.coverage(case.lens, starts, targets, clen)
    cov.set_scale(case.scale)
    fetched = cov.to_list()
    if store.name == "wide" and case.n <= 1024:
        assert max(int(c.max()) for c in fetched if c is not None) > 65535
    for stat in ("mean", "median"):
        ref, tol = reference(fetched, case.n, case.where, case.f1, case.f2, case.scale, case.kind, stat)
        outs = []
        for ctas in (KNOB if stat == "mean" else [None]):
            if ctas is None:
                monkeypatch.delenv("RCP_BIN_CTAS", raising=False)
            else:
                monkeypatch.setenv("RCP_BIN_CTAS", str(ctas))
            outs.append(bin_matrix(rb, cov, case, stat))
        monkeypatch.delenv("RCP_BIN_CTAS", raising=False)
        for ctas, o in zip(KNOB[1:], outs[1:]):
            assert np.array_equal(o.view(np.uint64), outs[0].view(np.uint64)), "RCP_BIN_CTAS=%d" % ctas
        assert_matches(outs[0], ref, tol, stat)


def device_call(rb, fn, shape, ld, offset, args):
    """fn(*args, ptr, ld, MEM_DEVICE) into a torch buffer of ld x cols (+ offset doubles) filled
    with a sentinel; returns (matrix, the padding and the leading guard)."""
    import torch
    from recoup_b200 import _lib
    R, ncol = shape
    buf = torch.full((offset + ld * ncol,), -123.25, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    _lib.check(fn(*args, buf.data_ptr() + 8 * offset, ld, _lib.MEM_DEVICE))
    _lib.check(_lib.lib.rcp_sync())
    host = buf.cpu().numpy()
    m = host[offset:].reshape(ncol, ld).T
    return m[:R], np.concatenate([host[:offset], m[R:].ravel()])


@pytest.mark.gpu
@pytest.mark.parametrize("ci", [2, 5, 11])
def test_bin_matrix_into_device_memory(store, ci):
    rb = store.rb
    from recoup_b200 import _lib
    case = BIN_CASES[ci]
    starts, targets, clen = targets_for(case.lens, case.n, case.where, case.f1, case.f2, case.kind, store.name)
    cov = store.coverage(case.lens, starts, targets, clen, check=False)
    cov.set_scale(case.scale)
    R = len(cov)
    w = _lib.WHERE[case.where]
    for stat in ("mean", "median"):
        want = bin_matrix(rb, cov, case, stat)
        for ld, offset in [(R + 6, 0), (R + 3, 1)]:
            args = (cov.handle, w, case.f1, case.f2, case.n, _lib.STAT[stat], _lib.INTERP["auto"], SEED,
                    _lib.SAMPLE_KIND[case.kind])
            got, pad = device_call(rb, _lib.lib.rcp_bin_matrix, (R, case.n), ld, offset, args)
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (stat, ld, offset)
            assert (pad == -123.25).all()


# ---- GPU: per-base matrices ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_cols", [3, 127, 128, 255, 256, 257])
def test_base_matrix_exact(store, n_cols):
    rb = store.rb
    from recoup_b200 import _lib
    R = 1000 + 7                                   # R % 32 != 0
    for where, f1, f2 in [("upstream", n_cols, 300), ("downstream", 1001, n_cols)]:
        lens = [None if i % 41 == 0 else n_cols + i % 9 for i in range(R)]
        starts, targets, clen = targets_for(lens, 1, "whole", 0, 0, "Rejection", store.name)
        cov = store.coverage(lens, starts, targets, clen)
        cov.set_scale(0.37)
        ref = np.zeros((R, n_cols))
        for r, c in enumerate(cov.to_list()):
            if c is not None:
                a, b = segment(c.shape[0], where, f1, f2)
                ref[r, :b - a] = 0.37 * c[a:b].astype(np.float64)
        got = np.asarray(rb.baseCoverageMatrix(cov, flank=(f1, f2), where=where))
        assert_matches(got, ref, np.zeros_like(ref), "%s host" % where)
        # odd leading dimension and a matrix one double off 16-byte alignment: scalar stores
        for ld, offset in [(R + 1, 0), (R + 2, 1)]:
            got, pad = device_call(rb, _lib.lib.rcp_base_matrix, (R, n_cols), ld, offset,
                                   (cov.handle, _lib.WHERE[where], f1, f2, n_cols))
            assert_matches(got, ref, np.zeros_like(ref), "%s ld %d offset %d" % (where, ld, offset))
            assert (pad == -123.25).all()


@pytest.mark.gpu
@pytest.mark.parametrize("storage", ["narrow", "wide"])
def test_base_matrix_past_one_launch_of_rows(rb, monkeypatch, storage):
    """2.2 M regions, 3 columns: base_matrix_kernel walks the rows in slabs of 2 097 120."""
    from recoup_b200 import _lib
    st = Store(storage, rb, monkeypatch)
    R = 2_200_000
    L = 3 + np.arange(R) % 4
    pos = 1 + np.concatenate([[0], np.cumsum(L + 1)[:-1]])
    clen = int(pos[-1] + L[-1] + 10)
    flat = hash8(np.arange(int(L.sum())) * 7 + 3)
    G = np.zeros(clen, dtype=np.int64)
    gidx = np.repeat(pos - 1, L) + (np.arange(int(L.sum())) - np.repeat(np.cumsum(L) - L, L))
    G[gidx] = flat
    s, e = level_reads(G)
    reads = rb.GRanges(np.zeros(s.shape[0], dtype=np.int32), s + 1, e + 1, strand=np.zeros(s.shape[0], np.int8),
                       seqlevels=["c0"], seqlengths=[clen])
    mask = rb.GRanges(np.zeros(R, dtype=np.int32), pos, pos + L - 1, strand=np.ones(R, np.int8), seqlevels=["c0"])
    if storage == "wide":
        monkeypatch.setenv("RCP_COVERAGE_WIDE", "1")
    cov = rb.calcCoverage(reads, mask)
    monkeypatch.delenv("RCP_COVERAGE_WIDE", raising=False)
    assert st.storage_bytes(cov) == (4 if storage == "wide" else 2)
    buf = np.zeros(int(L.sum()), dtype=np.int32)
    _lib.check(_lib.lib.rcp_coverage_fetch(cov.handle, 0, R, buf.ctypes.data_as(C.POINTER(C.c_int32)), buf.shape[0]))
    assert np.array_equal(buf, flat)
    got = np.asarray(rb.baseCoverageMatrix(cov, flank=(3, 3), where="upstream"))
    first = np.cumsum(L) - L
    ref = np.stack([flat[first + k] for k in range(3)], axis=1).astype(np.float64)
    for r0 in (BASE_SLAB_ROWS - 40, R - 40):
        assert np.array_equal(got[r0:r0 + 80], ref[r0:r0 + 80]), r0
    sample = np.random.default_rng(5).integers(0, R, size=20_000)
    assert np.array_equal(got[sample], ref[sample])
    assert np.array_equal(got.sum(axis=0), ref.sum(axis=0))
    assert np.array_equal(got, ref)


# ---- GPU: the fused coverage -> profile path ---------------------------------------------------
def fused_setup(rb, R, L, n, kind, pile=0):
    lens = [None if i % 29 == 3 else L for i in range(R)]
    starts, targets, clen = targets_for(lens, n, "whole", 0, 0, kind, "narrow")
    if pile:
        targets[1][L // 2] += pile                  # one base of one window
    G = genome_vector(starts, targets, clen, np.int64)
    s, e = level_reads(G)
    reads = rb.GRanges(np.zeros(s.shape[0], dtype=np.int32), s + 1, e + 1, strand=np.zeros(s.shape[0], np.int8),
                       seqlevels=["c0", "c1"], seqlengths=[clen, 1000])
    chrom, ms, me = mask_arrays(starts, [L] * R)
    mask = rb.GRanges(chrom, ms, me, strand=np.ones(R, np.int8), seqlevels=["c0", "c1"])
    return reads, mask, targets


@pytest.mark.gpu
@pytest.mark.parametrize("L,n,R,pile", [(1000, 1000, 600, 0), (1000, 999, 600, FUSED_SMALL + 1000),
                                        (31_000, 6000, 64, 0), (31_000, FUSED_MAX_BINS, 64, 0),
                                        (31_000, FUSED_MAX_BINS + 1, 64, 0)])
def test_fused_profile_exact_and_equal_to_two_stages(rb, L, n, R, pile):
    kind, scale = "Rounding", 0.37
    reads, mask, targets = fused_setup(rb, R, L, n, kind, pile)
    got, is_null = rb.coverageProfile(reads, mask, n, scale=scale, sample_kind=kind)
    got = np.asarray(got)
    cov = rb.calcCoverage(reads, mask)
    fetched = cov.to_list()
    assert_same_coverage(fetched, targets)
    assert np.array_equal(is_null, np.array([t is None for t in targets]))
    ref, tol = reference(fetched, n, "whole", 0, 0, scale, kind, "mean")
    assert not tol.any()
    assert_matches(got, ref, tol, "fused")
    cov.set_scale(scale)
    inp = [dict(name="s", coverage=cov)]
    rb.profileMatrix(inp, (0, 0), dict(flankBinSize=0, regionBinSize=n, sumStat="mean"), sample_kind=kind)
    two = np.asarray(inp[0]["profile"])
    assert np.array_equal(two.view(np.uint64), got.view(np.uint64))


# ---- GPU: limits -------------------------------------------------------------------------------
def pool_used():
    """cudaMemPoolAttrUsedMemCurrent of device 0's default pool (driver API)."""
    cu = C.CDLL("libcuda.so.1")
    dev, pool, val = C.c_int(0), C.c_void_p(0), C.c_uint64(0)
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    assert cu.cuMemPoolGetAttribute(pool, 7, C.byref(val)) == 0      # CU_MEMPOOL_ATTR_USED_MEM_CURRENT
    return val.value


@pytest.mark.gpu
def test_bin_count_limits_fail_cleanly(store):
    rb = store.rb
    from recoup_b200 import _lib
    lens = [MAX_BINS + 700 + i for i in range(6)] + [None, 100]          # the last window is short
    starts, targets, clen = targets_for(lens, 7, "whole", 0, 0, "Rejection", store.name)
    cov = store.coverage(lens, starts, targets, clen, check=False)
    for stat in ("mean", "median"):
        for n in (MAX_BINS + 1, INTERP_MAX_BINS + 1, 6000):
            _lib.check(_lib.lib.rcp_sync())
            before = pool_used()
            with pytest.raises(_lib.RecoupError) as e:
                rb.binCoverageMatrix(cov, binSize=n, stat=stat)
            assert e.value.code == _lib.RCP_ERR_UNSUPPORTED, (stat, n, str(e.value))
            _lib.check(_lib.lib.rcp_sync())
            assert pool_used() == before, (stat, n)
    # without the short window every count up to the limit works
    lens2 = lens[:6]
    starts2, targets2, clen2 = targets_for(lens2, MAX_BINS, "whole", 0, 0, "Rejection", store.name)
    cov2 = store.coverage(lens2, starts2, targets2, clen2)
    fetched = cov2.to_list()
    for stat in ("mean", "median"):
        for n in (6000, MAX_BINS):
            ref, tol = reference(fetched, n, "whole", 0, 0, 1.0, "Rejection", stat)
            assert_matches(rb.binCoverageMatrix(cov2, binSize=n, stat=stat), ref, tol, "%s %d" % (stat, n))
