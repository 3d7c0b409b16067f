"""ORACLE -- CPU restatement of recoup's coverage -> profile-matrix path (numpy).

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this package; the product (recoup_b200/) never does.

PARITY UNPINNED: the reference is interpreted R whose arithmetic lives in un-vendored
Bioconductor/base-R packages (GenomicRanges, IRanges, S4Vectors, plyr, stats; DESCRIPTION:7-17,
no versions pinned), R is not installed in this image, and the reference's own tests assert no
numbers (inst/unitTests/test_recoup.R:28-31).  This restatement therefore follows the reference's
R source line by line and the *documented* semantics of the third-party calls, and is pinned by
(1) the R RNG known answers (oracle/r_rng.py), (2) the input fixture decoded from
data/recoup_test_data.rda and the invariants SURVEY.md section 4 derives from it, and (3) a
brute-force definition of coverage (`cov[p] = #{reads: start <= p <= end}`) used in the property
tests.

Conventions: coordinates are 1-based closed [start, end]; strand is +1 / -1 / 0 ('*');
a coverage is a python list with one entry per region: an int64 numpy vector (5'->3' oriented)
or None (R NULL).  File:line citations are relative to /root/reference/.
"""
import math

import numpy as np

from .r_rng import RRandom


# --------------------------------------------------------------------------------------------
# Region geometry                                                         R/ranges.R:67-100
# --------------------------------------------------------------------------------------------
def _promoters(start, end, strand, upstream, downstream):
    """GenomicRanges::promoters(): '+'/'*' anchor at start, '-' anchor at end."""
    minus = strand < 0
    s = np.where(minus, end - downstream + 1, start - upstream)
    e = np.where(minus, end + upstream, start + downstream - 1)
    return s, e


def _resize(start, end, strand, width, fix="start"):
    """GenomicRanges::resize(): fix='start' keeps the 5' end ('-' keeps `end`)."""
    minus = strand < 0
    keep_start = ~minus if fix == "start" else minus
    s = np.where(keep_start, start, end - width + 1)
    e = np.where(keep_start, start + width - 1, end)
    return s, e


def get_regional_ranges(start, end, strand, region, flank):
    """getRegionalRanges (R/ranges.R:67-91)."""
    start = np.asarray(start, dtype=np.int64)
    end = np.asarray(end, dtype=np.int64)
    strand = np.asarray(strand, dtype=np.int64)
    f1, f2 = int(flank[0]), int(flank[1])
    w = end - start + 1
    if region == "custom":
        region = "tss" if np.all(w == 1) else "genebody"      # ranges.R:81-89
    if region == "genebody":                                  # ranges.R:69-73
        s, e = _promoters(start, end, strand, f1, 0)
        return _resize(s, e, strand, w + f1 + f2, "start")
    if region == "tss":                                       # ranges.R:74-76
        return _promoters(start, end, strand, f1, f2)
    if region == "tes":                                       # ranges.R:77-80
        s, e = _resize(start, end, strand, 1, "end")
        return _promoters(s, e, strand, f1, f2)
    raise ValueError("unknown region type %r" % (region,))


def get_flanking_ranges(start, end, strand, flank, direction):
    """getFlankingRanges (R/ranges.R:93-100): promoters(x, flank, 0) / flank(x, flank, start=FALSE)."""
    start = np.asarray(start, dtype=np.int64)
    end = np.asarray(end, dtype=np.int64)
    strand = np.asarray(strand, dtype=np.int64)
    if direction == "upstream":
        return _promoters(start, end, strand, int(flank), 0)
    if direction == "downstream":
        minus = strand < 0
        s = np.where(minus, start - flank, end + 1)
        e = np.where(minus, start - 1, end + flank)
        return s, e
    raise ValueError(direction)


# --------------------------------------------------------------------------------------------
# Reads container
# --------------------------------------------------------------------------------------------
class Reads:
    """Decoded reads (the GRanges `input` of calcCoverage): chrom id, start, end, strand.
    `chrom_len[c]` is seqlengths(); -1 encodes NA."""

    def __init__(self, chrom, start, end, strand, chrom_len):
        self.chrom = np.asarray(chrom, dtype=np.int64)
        self.start = np.asarray(start, dtype=np.int64)
        self.end = np.asarray(end, dtype=np.int64)
        self.strand = np.asarray(strand, dtype=np.int64)
        self.chrom_len = np.asarray(chrom_len, dtype=np.int64)
        n = self.start.shape[0]
        assert self.chrom.shape == (n,) and self.end.shape == (n,) and self.strand.shape == (n,)

    def __len__(self):
        return self.start.shape[0]

    def subset(self, keep):
        return Reads(self.chrom[keep], self.start[keep], self.end[keep], self.strand[keep],
                     self.chrom_len)


def extend_fragments(start, end, strand, frag_len, chrom, chrom_len):
    """A0 (SURVEY 8a): fragment extension named by north_star but ABSENT from the reference
    (R/ranges.R:1-65 has none).  Semantics defined as GenomicRanges
    `trim(resize(reads, fragLen, fix="start"))`: '+'/'*' keep start, '-' keep end; then clip
    into [1, seqlength]."""
    start = np.asarray(start, dtype=np.int64)
    end = np.asarray(end, dtype=np.int64)
    strand = np.asarray(strand, dtype=np.int64)
    s, e = _resize(start, end, strand, int(frag_len), "start")
    clen = np.asarray(chrom_len, dtype=np.int64)[np.asarray(chrom, dtype=np.int64)]
    s = np.maximum(s, 1)
    e = np.where(clen > 0, np.minimum(e, clen), e)
    return s, e


# --------------------------------------------------------------------------------------------
# Coverage                                                              R/coverage.R:126-226
# --------------------------------------------------------------------------------------------
def _strand_compatible(read_strand, region_strand):
    """findOverlaps(ignore.strand=FALSE): '*' matches anything, otherwise strands must agree."""
    if region_strand == 0:
        return np.ones(read_strand.shape, dtype=bool)
    return (read_strand == region_strand) | (read_strand == 0)


def _index_subscript(cov_len, idx):
    """`Rle[idx]` with R / S4Vectors subscript rules (coverage.R:206,209 inside tryCatch).
    Returns the kept 1-based indices or None when R would raise (=> NULL coverage):
    any index beyond the vector -> 'subscript contains out-of-bounds indices'; negative mixed
    with positive -> error; zeros are silently dropped."""
    if idx.size == 0:
        return idx
    if idx.max() > cov_len:
        return None
    if idx.min() < 0:
        if idx.max() > 0:
            return None
        # all non-positive: R would *drop* those elements; unreachable through recoup because
        # such a window cannot overlap a read (reads start at >= 1).
        return None
    return idx[idx != 0]


def coverage_from_ranges(reads, chrom, starts, ends, strands, ignore_strand=True):
    """coverageFromRanges (R/coverage.R:176-226) for ONE mask element.

    `starts/ends/strands` are scalars-in-arrays for a GRanges element, or all exons of one gene
    for a GRangesList element (chromosome/strand taken from the FIRST range, coverage.R:182,185).
    Returns int64 vector or None.
    """
    starts = np.atleast_1d(np.asarray(starts, dtype=np.int64))
    ends = np.atleast_1d(np.asarray(ends, dtype=np.int64))
    strands = np.atleast_1d(np.asarray(strands, dtype=np.int64))
    on_chr = reads.chrom == chrom
    if not on_chr.any():                                   # coverage.R:189,194-197
        return None
    rs, re_, rst = reads.start[on_chr], reads.end[on_chr], reads.strand[on_chr]
    # findOverlaps(x, reads): one hit per (range of x, read) pair -> a read overlapping k exons
    # is selected k times (coverage.R:190-192); zero-width ranges never hit.
    mult = np.zeros(rs.shape[0], dtype=np.int64)
    for s, e, st in zip(starts, ends, strands):
        if e < s:
            continue
        hit = (rs <= e) & (re_ >= s)
        if not ignore_strand:
            hit &= _strand_compatible(rst, int(st))
        mult += hit
    sel = mult > 0
    if not sel.any():                                      # coverage.R:198,224-225
        return None
    # coverage(y$reads)[[chr]]: whole-chromosome integer vector; length = seqlength when known,
    # else the largest end among the selected reads (coverage.R:201)
    clen = int(reads.chrom_len[chrom])
    cov_len = clen if clen > 0 else int(re_[sel].max())
    # i2k (coverage.R:202-209)
    idx = np.concatenate([np.arange(s, e + 1, dtype=np.int64) for s, e in zip(starts, ends)])
    idx = _index_subscript(cov_len, idx)
    if idx is None:                                        # tryCatch -> NULL (coverage.R:217-222)
        return None
    lo, hi = (int(idx.min()), int(idx.max())) if idx.size else (1, 0)
    diff = np.zeros(max(hi - lo + 2, 1), dtype=np.int64)
    s_sel, e_sel, m_sel = rs[sel], re_[sel], mult[sel]
    a = np.clip(s_sel, lo, hi + 1) - lo
    b = np.clip(e_sel + 1, lo, hi + 1) - lo
    np.add.at(diff, a, m_sel)
    np.add.at(diff, b, -m_sel)
    cov = np.cumsum(diff)[:-1]
    out = cov[idx - lo] if idx.size else np.zeros(0, dtype=np.int64)
    if int(strands[0]) < 0:                                # coverage.R:210-215
        out = out[::-1]
    return np.ascontiguousarray(out)


def calc_coverage(reads, mask, strand=None, ignore_strand=True):
    """calcCoverage (R/coverage.R:126-174) for in-memory reads.

    `mask` is a dict with chrom/start/end/strand arrays (GRanges) or additionally `ptr`
    (GRangesList: ranges ptr[i]:ptr[i+1] belong to element i).  Returns a list of vectors/None.
    """
    if strand is not None:                                 # coverage.R:141-144
        reads = reads.subset(reads.strand == int(strand))
    chrom = np.asarray(mask["chrom"], dtype=np.int64)
    ms = np.asarray(mask["start"], dtype=np.int64)
    me = np.asarray(mask["end"], dtype=np.int64)
    mst = np.asarray(mask["strand"], dtype=np.int64)
    out = []
    if "ptr" in mask:
        ptr = np.asarray(mask["ptr"], dtype=np.int64)
        for i in range(ptr.shape[0] - 1):
            a, b = int(ptr[i]), int(ptr[i + 1])
            if b <= a:      # empty element: seqnames(x)[1] is NA -> "not found" -> NULL
                out.append(None)
                continue
            out.append(coverage_from_ranges(reads, int(chrom[a]), ms[a:b], me[a:b], mst[a:b],
                                            ignore_strand))
    else:
        for i in range(ms.shape[0]):
            out.append(coverage_from_ranges(reads, int(chrom[i]), ms[i:i + 1], me[i:i + 1],
                                            mst[i:i + 1], ignore_strand))
    return out


def coverage_ref(reads, genome, region, flank, strand=None, ignore_strand=True):
    """coverageRef (R/coverage.R:1-77): tss/tes/1-bp custom and genebody/wide custom all reduce to
    calcCoverage over getRegionalRanges(...)."""
    s, e = get_regional_ranges(genome["start"], genome["end"], genome["strand"], region, flank)
    mask = dict(chrom=genome["chrom"], start=s, end=e, strand=genome["strand"])
    return calc_coverage(reads, mask, strand, ignore_strand)


def coverage_rna_ref(reads, exons, genes, flank, strand=None, ignore_strand=True):
    """coverageRnaRef (R/coverage.R:79-124).  `exons` = GRangesList dict (with ptr), `genes` =
    helperRanges dict.  Reproduces the reference's flank quirks: width 1 when flank[1]==0 and
    the right flank tested against flank[1] (coverage.R:84-91)."""
    f1, f2 = int(flank[0]), int(flank[1])
    lw = 1 if f1 == 0 else f1
    rw = 1 if f1 == 0 else f2
    ls, le = get_flanking_ranges(genes["start"], genes["end"], genes["strand"], lw, "upstream")
    rs, re_ = get_flanking_ranges(genes["start"], genes["end"], genes["strand"], rw, "downstream")
    center = calc_coverage(reads, exons, strand, ignore_strand)
    left = calc_coverage(reads, dict(chrom=genes["chrom"], start=ls, end=le,
                                     strand=genes["strand"]), strand, ignore_strand)
    right = calc_coverage(reads, dict(chrom=genes["chrom"], start=rs, end=re_,
                                      strand=genes["strand"]), strand, ignore_strand)
    out = []
    for l, c, r in zip(left, center, right):               # coverage.R:115-120
        if l is None or c is None or r is None:
            out.append(None)
        else:
            out.append(np.concatenate([l, c, r]))
    return out


# --------------------------------------------------------------------------------------------
# stats::spline(method="fmm")  -- base R, not vendored; published FMM algorithm
# (Forsythe, Malcolm & Moler 1977; R src/library/stats/src/splines.c fmm_spline/spline_eval)
# --------------------------------------------------------------------------------------------
def _fmm_coef(x, y):
    n = len(x)
    b = [0.0] * n
    c = [0.0] * n
    d = [0.0] * n
    if n < 2:
        return b, c, d
    if n < 3:
        t = y[1] - y[0]
        b[0] = t / (x[1] - x[0])
        b[1] = b[0]
        return b, c, d
    nm1 = n - 1
    d[0] = x[1] - x[0]
    c[1] = (y[1] - y[0]) / d[0]
    for i in range(1, nm1):
        d[i] = x[i + 1] - x[i]
        b[i] = 2.0 * (d[i - 1] + d[i])
        c[i + 1] = (y[i + 1] - y[i]) / d[i]
        c[i] = c[i + 1] - c[i]
    b[0] = -d[0]
    b[n - 1] = -d[n - 2]
    c[0] = c[n - 1] = 0.0
    if n > 3:
        c[0] = c[2] / (x[3] - x[1]) - c[1] / (x[2] - x[0])
        c[n - 1] = c[n - 2] / (x[n - 1] - x[n - 3]) - c[n - 3] / (x[n - 2] - x[n - 4])
        c[0] = c[0] * d[0] * d[0] / (x[3] - x[0])
        c[n - 1] = -c[n - 1] * d[n - 2] * d[n - 2] / (x[n - 1] - x[n - 4])
    for i in range(1, n):
        t = d[i - 1] / b[i - 1]
        b[i] = b[i] - t * d[i - 1]
        c[i] = c[i] - t * c[i - 1]
    c[n - 1] = c[n - 1] / b[n - 1]
    for i in range(n - 2, -1, -1):
        c[i] = (c[i] - d[i] * c[i + 1]) / b[i]
    b[n - 1] = (y[n - 1] - y[n - 2]) / d[n - 2] + d[n - 2] * (c[n - 2] + 2.0 * c[n - 1])
    for i in range(nm1):
        b[i] = (y[i + 1] - y[i]) / d[i] - d[i] * (c[i + 1] + 2.0 * c[i])
        d[i] = (c[i + 1] - c[i]) / d[i]
        c[i] = 3.0 * c[i]
    c[n - 1] = 3.0 * c[n - 1]
    d[n - 1] = d[n - 2]
    return b, c, d


def r_spline(yv, n):
    """`spline(yv, n=n)$y`: x = seq_along(yv), xout = seq.int(1, L, length.out=n), method fmm."""
    L = len(yv)
    y = [float(v) for v in yv]
    x = [float(i + 1) for i in range(L)]
    b, c, d = _fmm_coef(x, y)
    if n == 1:
        xout = [1.0]
    else:
        by = (float(L) - 1.0) / float(n - 1) if n > 2 else 0.0
        xout = [1.0 + i * by for i in range(n)]
        xout[0] = 1.0
        xout[n - 1] = float(L)
    out = np.empty(n, dtype=np.float64)
    i = 0
    for l, ul in enumerate(xout):
        if ul < x[i] or (i < L - 1 and x[i + 1] < ul):
            i, j = 0, L
            while True:
                k = (i + j) // 2
                if ul < x[k]:
                    j = k
                else:
                    i = k
                if j <= i + 1:
                    break
        dx = ul - x[i]
        out[l] = y[i] + dx * (b[i] + dx * (c[i] + dx * d[i]))
    return out


# --------------------------------------------------------------------------------------------
# splitVector                                                              R/util.R:15-85
# --------------------------------------------------------------------------------------------
def _neighborhood(x, n, seed, sample_kind):
    """util.R:24-38 / 54-68."""
    L = len(x)
    if L < 4 or n < 6:
        raise ValueError("neighborhood interpolation needs length(x) >= 4 and n >= 6 "
                         "(R's sample() would stop())")
    y = np.full(n, np.nan)
    rng = RRandom(seed, sample_kind)
    y[0:2] = x[0:2]
    y[n - 2:n] = x[L - 2:L]
    pool = list(range(3, n - 1))                             # 3:(n-2)
    picks = rng.sample_int(len(pool), L - 4)
    orig_pos = sorted(pool[p - 1] for p in picks)
    if orig_pos:
        y[np.asarray(orig_pos) - 1] = x[2:L - 2]
    na = np.flatnonzero(np.isnan(y)) + 1                     # 1-based
    fill = []
    for z in na:
        ii = np.array([z - 2, z - 1, z + 1, z + 2]) - 1
        vals = y[ii]
        vals = vals[~np.isnan(vals)]
        fill.append(vals.mean() if vals.size else np.nan)
    y[na - 1] = fill
    return y


def bin_layout(L, n, seed=42, sample_kind="Rejection"):
    """util.R:74-80: sizes of the n contiguous bins of a length-L vector (L >= n)."""
    bin_size = L // n
    dif = L - bin_size * n
    fac = np.full(n, bin_size, dtype=np.int64)
    add = RRandom(seed, sample_kind).sample_int(n, dif)
    fac[np.asarray(add, dtype=np.int64) - 1] += 1
    return fac


def split_vector(x, n, interp="auto", stat="mean", seed=42, sample_kind="Rejection"):
    """splitVector + llply(S, stat) (R/util.R:15-85): returns float64[n]."""
    x = np.asarray(x, dtype=np.float64)
    L = x.shape[0]
    if L < n:
        if interp == "auto":                                 # util.R:21-44
            if (n - L) / n < 0.2:
                x = _neighborhood(x, n, seed, sample_kind)
            else:
                x = np.maximum(r_spline(x, n), 0.0)
        elif interp == "spline":                             # util.R:45-48
            x = np.maximum(r_spline(x, n), 0.0)
        elif interp == "neighborhood":                       # util.R:53-69
            x = _neighborhood(x, n, seed, sample_kind)
        else:
            # util.R:49 -- the switch label is misspelt 'inear', so interpolation="linear"
            # leaves x short; factor() then drops the empty bins and rbind recycles rows.
            raise ValueError("interpolation=%r hits dead code in the reference "
                             "(R/util.R:49); not reproduced" % (interp,))
        L = n
    fac = bin_layout(L, n, seed, sample_kind)
    edges = np.concatenate([[0], np.cumsum(fac)])
    out = np.empty(n, dtype=np.float64)
    for i in range(n):
        seg = x[edges[i]:edges[i + 1]]
        if stat == "mean":
            out[i] = seg.sum() / seg.shape[0] if seg.shape[0] else np.nan
        elif stat == "median":
            out[i] = np.median(seg) if seg.shape[0] else np.nan
        else:
            raise ValueError(stat)
    return out


# --------------------------------------------------------------------------------------------
# Profile matrix                                                         R/profile.R:1-212
# --------------------------------------------------------------------------------------------
def _slice_where(c, flank, where):
    """profile.R:127-140,166-188 slices of one non-NULL coverage vector."""
    f1, f2 = int(flank[0]), int(flank[1])
    nr = c.shape[0]
    if where == "center":
        return c[f1:nr - f2]
    if where == "upstream":
        return c[0:f1]
    if where == "downstream":
        return c[nr - f2:nr]
    raise ValueError(where)


def bin_coverage_matrix(cvrg, bin_size=1000, stat="mean", interpolation="auto", flank=None,
                        where="center", seed=42, sample_kind="Rejection"):
    """binCoverageMatrix (R/profile.R:153-212)."""
    rows = []
    for c in cvrg:
        if c is None:
            rows.append(np.zeros(bin_size))                  # profile.R:191-197 + splitVector
            continue
        x = c if flank is None else _slice_where(c, flank, where)
        rows.append(split_vector(x, bin_size, interpolation, stat, seed, sample_kind))
    return np.vstack(rows) if rows else np.zeros((0, bin_size))


def base_coverage_matrix(cvrg, flank=None, where="upstream"):
    """baseCoverageMatrix (R/profile.R:100-151)."""
    if flank is None:
        size = 0
        for c in cvrg:                                       # profile.R:103-111
            if c is not None:
                size = c.shape[0]
                break
        rows = [np.zeros(size) if c is None else c.astype(np.float64) for c in cvrg]
    else:
        size = int(flank[0]) if where == "upstream" else int(flank[1])
        rows = [np.zeros(size) if c is None else _slice_where(c, flank, where).astype(np.float64)
                for c in cvrg]
    return np.vstack(rows) if rows else np.zeros((0, size))


def r_round(x):
    """R's round(): IEC 60559 half-to-even (python's round() agrees)."""
    return int(round(x))


def have_equal_lengths(cvrg):
    """profile.R:6-10: lengths without the zero-length (NULL) entries, all equal to the first."""
    lens = [c.shape[0] for c in cvrg if c is not None and c.shape[0] > 0]
    return all(l == lens[0] for l in lens) if lens else True


def profile_matrix(cvrg, flank, bin_params, seed=42, sample_kind="Rejection",
                   equal_lengths=None):
    """profileMatrix (R/profile.R:1-98) for one sample's coverage list.

    `bin_params` keys: flankBinSize, regionBinSize, sumStat, interpolation.  `equal_lengths`
    lets a caller pass the decision made on the FIRST sample (profile.R:6 uses input[[1]] only).
    """
    fbs = int(bin_params.get("flankBinSize", 0))
    rbs = int(bin_params.get("regionBinSize", 0))
    stat = bin_params.get("sumStat", "mean")
    interp = bin_params.get("interpolation", "auto")
    f1, f2 = int(flank[0]), int(flank[1])
    if equal_lengths is None:
        equal_lengths = have_equal_lengths(cvrg)
    if equal_lengths:                                        # profile.R:83-96
        if rbs != 0:
            # NB interpolation is NOT forwarded here (profile.R:88-90) -> default "auto"
            return bin_coverage_matrix(cvrg, rbs, stat, "auto", None, "center", seed, sample_kind)
        return base_coverage_matrix(cvrg)
    center = bin_coverage_matrix(cvrg, rbs, stat, interp, (f1, f2), "center", seed, sample_kind)
    left = right = None
    if fbs != 0:                                             # profile.R:25-57
        tot = float(f1 + f2)
        if f1 != 0:
            left = bin_coverage_matrix(cvrg, r_round(2 * fbs * (f1 / tot)), stat, interp,
                                       (f1, f2), "upstream", seed, sample_kind)
        if f2 != 0:
            right = bin_coverage_matrix(cvrg, r_round(2 * fbs * (f2 / tot)), stat, interp,
                                        (f1, f2), "downstream", seed, sample_kind)
    else:                                                    # profile.R:58-77
        if f1 != 0:
            left = base_coverage_matrix(cvrg, (f1, f2), "upstream")
        if f2 != 0:
            right = base_coverage_matrix(cvrg, (f1, f2), "downstream")
    parts = [p for p in (left, center, right) if p is not None]
    return np.hstack(parts)                                  # profile.R:78


def linear_factors(lib_sizes, normalize="linear", sample_to=None):
    """calcLinearFactors (R/util.R:349-362)."""
    lib = np.asarray(lib_sizes, dtype=np.float64)
    if normalize in ("linear", "downsample"):
        return lib.min() / lib
    if normalize == "sampleto":
        return float(sample_to) / lib
    raise ValueError(normalize)


# --------------------------------------------------------------------------------------------
# Brute-force definition used as the property-test ground truth (SURVEY 8c item 3)
# --------------------------------------------------------------------------------------------
# --------------------------------------------------------------------------------------------
# Read import after decoding                                        R/ranges.R:1-65,111-134
# --------------------------------------------------------------------------------------------
def splice_remove(start, end, sq=0.75):
    """readBam(sa = "remove") (ranges.R:125-133): qu = quantile(width(reads), sq); the reads wider
    than qu are excluded.  Returns the boolean keep mask and qu."""
    width = np.asarray(end, dtype=np.int64) - np.asarray(start, dtype=np.int64) + 1
    qu = float(r_quantile7(width, [sq])[0])
    return ~(width > qu), qu


def downsample_indices(lib_sizes, normalize, seed=42, sample_to=1000000, sample_kind="Rejection"):
    """preprocessRanges normalize = "downsample" / "sampleto" (ranges.R:31-63): ONE set.seed, then
    sort(sample(libSize, s)) per sample, s = min(libSizes) or sampleTo.  1-based indices;
    None for "none" / "linear"."""
    if normalize in ("none", "linear"):
        return [None for _ in lib_sizes]
    s = min(lib_sizes) if normalize == "downsample" else int(sample_to)
    rng = RRandom(seed, sample_kind)
    return [np.sort(np.asarray(rng.sample_int(int(n), s), dtype=np.int64)) for n in lib_sizes]


# --------------------------------------------------------------------------------------------
# Consumers of the profile matrix                                  R/plot.R:513-545,949-1150
# --------------------------------------------------------------------------------------------
def r_mean(x):
    """base R mean(): long-double sum / n, then one refinement pass (summary.c, real_mean)."""
    x = np.asarray(x, dtype=np.longdouble)
    n = x.shape[0]
    s = x.sum() / n
    s += (x - s).sum() / n
    return float(s)


def r_median(x):
    x = np.sort(np.asarray(x, dtype=np.float64))
    n = x.shape[0]
    if n and np.isnan(x[-1]):
        return float("nan")
    return float(x[(n - 1) // 2]) if n % 2 else float((x[n // 2 - 1] + x[n // 2]) / 2.0)


def plot_profile(profile, avgfun="mean", scale="natural"):
    """calcPlotProfiles without smoothing (plot.R:976-990): apply(x$profile, 2, avgfun) and the
    band  profile +- sd  (mean) or  +- mad  (median; stats::mad constant 1.4826), after
    x <- log2(x + 1) when signalScale is "log2" (plot.R:978-981)."""
    x = np.asarray(profile, dtype=np.float64)
    if scale == "log2":
        x = np.log2(x + 1.0)
    n = x.shape[0]
    center = np.empty(x.shape[1])
    spread = np.empty(x.shape[1])
    for j in range(x.shape[1]):
        col = x[:, j]
        if avgfun == "mean":
            m = r_mean(col)
            center[j] = m
            d = col.astype(np.longdouble) - np.longdouble(m)
            spread[j] = float(np.sqrt((d * d).sum() / (n - 1))) if n > 1 else float("nan")
        else:
            m = r_median(col)
            center[j] = m
            spread[j] = 1.4826 * r_median(np.abs(col - m))
    return {"profile": center, "upper": center + spread, "lower": center - spread}


def row_order_values(profile, what):
    """apply(x$profile, 1, sum | max | mean) (plot.R:1080, 1122-1129, 1144); `what` is the
    prefix of orderBy$what ("sum", "max", "avg")."""
    x = np.asarray(profile, dtype=np.float64)
    if what == "sum":
        return np.array([float(np.asarray(r, dtype=np.longdouble).sum()) for r in x])
    if what == "max":
        return x.max(axis=1)
    if what == "avg":
        return np.array([r_mean(r) for r in x])
    raise ValueError(what)


def r_sort_index(v, decreasing=False):
    """sort(v, decreasing, index.return=TRUE)$ix (plot.R:1100-1103): 1-based, NA dropped, ties in
    input order both ways (order(method = "radix"), the default since R 3.3)."""
    v = np.asarray(v, dtype=np.float64)
    keep = np.flatnonzero(~np.isnan(v))
    key = -v[keep] if decreasing else v[keep]
    return keep[np.argsort(key + 0.0, kind="stable")] + 1


def r_quantile7(x, probs):
    """stats::quantile(x, probs, type = 7) (plot.R:519,536), in quantile.default's own
    arithmetic: index <- 1 + max(n - 1, 0) * probs, lo <- floor(index), 1-based reads,
    h <- index - lo.  Adding the 1 before taking h rounds h differently from (n - 1) * p - lo:
    quantile(c(0, 1), 0.1) is 0.10000000000000009, not 0.1."""
    x = np.sort(np.asarray(x, dtype=np.float64).ravel())
    if x.shape[0] and np.isnan(x[-1]):
        raise ValueError("missing values and NaN's not allowed if 'na.rm' is FALSE")
    n = x.shape[0]
    out = []
    for p in np.atleast_1d(probs):
        index = 1.0 + max(n - 1, 0) * float(p)
        lo, hi = int(math.floor(index)), int(math.ceil(index))
        q = x[lo - 1]
        h = index - lo
        if index > lo and x[hi - 1] != q:
            q = (1.0 - h) * q + h * x[hi - 1]
        out.append(float(q))
    return np.array(out)


def brute_coverage(read_start, read_end, lo, hi):
    """cov[p] = #{reads: start <= p <= end} for p in [lo, hi] -- O(N * L), tiny inputs only."""
    out = np.zeros(hi - lo + 1, dtype=np.int64)
    for s, e in zip(read_start, read_end):
        a, b = max(int(s), lo), min(int(e), hi)
        if a <= b:
            out[a - lo:b - lo + 1] += 1
    return out
