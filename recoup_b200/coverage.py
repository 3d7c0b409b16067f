"""Host mirror of /root/reference/R/coverage.R over librecoup_b200.so.

Same names, argument meaning and error behaviour as the reference's closures:

    calcCoverage(input, mask, strand=NULL, ignore.strand=TRUE, rc=NULL)      coverage.R:126-174
    coverageRef(input, genomeRanges, region, flank, strandedParams, ...)     coverage.R:1-77
    coverageRnaRef(input, genomeRanges, helperRanges, flank, ...)            coverage.R:79-124

`rc` (fraction of cores for mclapply, util.R:364-382) is accepted and ignored: the per-region
map runs as a CUDA grid.  All arithmetic happens in the CUDA library; this file only moves
arrays across the C ABI.  BigWig input (coverageFromBigWig, coverage.R:228-322) runs on the device
too: the track is loaded with readers.readBigWig and painted into the windows by
rcp_signal_coverage; its coverage holds float32 values.  BAM file paths stay outside this path:
pass the decoded ranges (readers.readBam).
"""
import ctypes as C
import os
import re
import weakref

import numpy as np

from . import _lib
from .ranges import GRanges, GRangesList, getFlankingRanges, getRegionalRanges, strand_to_code

_lib_check = _lib.check


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _message(*parts):
    # the reference reports progress with message(); keep it quiet unless asked
    if _VERBOSE:
        print("".join(str(p) for p in parts))


_VERBOSE = False


def set_verbose(flag):
    global _VERBOSE
    _VERBOSE = bool(flag)


# ------------------------------------------------------------------------------------------------
# device-resident objects
# ------------------------------------------------------------------------------------------------
def _seqlengths(gr):
    """seqlengths(gr) as int64; unknown lengths (None, NaN, <= 0: R's NA) travel as -1: the coverage
    vector of such a chromosome ends at the last overlapping read (coverage.R:201)."""
    if gr.seqlengths is None:
        return np.full(max(len(gr.seqlevels), 1), -1, dtype=np.int64)
    sl = np.asarray(gr.seqlengths)
    if sl.dtype.kind == "O":
        sl = np.asarray([np.nan if v is None else v for v in sl.tolist()], dtype=np.float64)
    if sl.dtype.kind == "f":
        sl = np.where(np.isnan(sl), -1, sl)
    sl = np.ascontiguousarray(sl, dtype=np.int64)
    return np.where(sl <= 0, -1, sl)


class DeviceReads:
    """Device index of one sample's reads (rcp_reads_load)."""

    def __init__(self, gr, frag_len=0, use_runs=None):
        """use_runs: send the seqnames as runs (rcp_reads_load_rle); default: when the GRanges
        holds them as an Rle with fewer than n / 2 runs."""
        _lib.ensure_init()
        h = C.c_int(0)
        if getattr(gr, "decoded_handle", None) is not None:
            # decoded on the device (readers.DecodedGRanges): no host round trip
            clen = _seqlengths(gr)
            _lib_check(_lib.lib.rcp_reads_load_decoded(gr.decoded_handle, clen.shape[0],
                                                       clen.ctypes.data_as(C.POINTER(C.c_int64)), int(frag_len),
                                                       C.byref(h)))
            self.handle = h.value
            self.n = len(gr)
            self.seqlevels = list(gr.seqlevels)
            self._fin = weakref.finalize(self, _free_reads, self.handle)
            return
        if getattr(gr, "parent", None) is not None:
            # a selection of another GRanges (preprocess.SelectedGRanges): the device applies it
            p = gr.parent
            if getattr(p, "decoded_handle", None) is not None:
                # a selection of reads decoded on the device: nothing but the index crosses PCIe
                clen = _seqlengths(gr)
                n_kept = C.c_int64(0)
                k = 0 if gr.idx is None else gr.idx.shape[0]
                _lib_check(_lib.lib.rcp_reads_load_decoded_select(
                    p.decoded_handle, -1.0 if gr.max_width is None else float(gr.max_width), k,
                    None if gr.idx is None else _ptr(gr.idx), clen.shape[0],
                    clen.ctypes.data_as(C.POINTER(C.c_int64)), int(frag_len), C.byref(n_kept), C.byref(h)))
                self.handle = h.value
                self.n = len(gr)
                self.seqlevels = list(gr.seqlevels)
                self._fin = weakref.finalize(self, _free_reads, self.handle)
                return
            arr = [np.ascontiguousarray(a, dtype=t) for a, t in
                   ((p.seqnames, np.int32), (p.start, np.int32), (p.end, np.int32), (p.strand, np.int8))]
            clen = _seqlengths(gr)
            n_kept = C.c_int64(0)
            k = 0 if gr.idx is None else gr.idx.shape[0]
            _lib_check(_lib.lib.rcp_reads_load_select(
                len(p), _ptr(arr[0]), _ptr(arr[1]), _ptr(arr[2]), _ptr(arr[3]),
                -1.0 if gr.max_width is None else float(gr.max_width), k,
                None if gr.idx is None else _ptr(gr.idx), clen.shape[0],
                clen.ctypes.data_as(C.POINTER(C.c_int64)), int(frag_len), _lib.MEM_HOST,
                C.byref(n_kept), C.byref(h)))
            self.handle = h.value
            self.n = len(gr)
            self.seqlevels = list(gr.seqlevels)
            self._fin = weakref.finalize(self, _free_reads, self.handle)
            return
        start = np.ascontiguousarray(gr.start, dtype=np.int32)
        strand = np.ascontiguousarray(gr.strand, dtype=np.int8)
        clen = _seqlengths(gr)
        clen_p = clen.ctypes.data_as(C.POINTER(C.c_int64))
        rle = gr.seqnames_rle
        if use_runs is None:
            use_runs = rle is not None and len(gr) < 2**32 - 16 and rle.nrun * 2 < len(gr)
        fixed = getattr(gr, "fixed_width", None)
        if fixed is not None:
            # one width for every read: start (+ strand) only cross PCIe
            if use_runs:
                run_chrom = np.ascontiguousarray(rle.values, dtype=np.int32)
                run_len = np.ascontiguousarray(rle.lengths, dtype=np.int32)
                _lib_check(_lib.lib.rcp_reads_load_width(len(gr), None, rle.nrun, _ptr(run_chrom), _ptr(run_len),
                                                         _ptr(start), int(fixed), _ptr(strand), clen.shape[0],
                                                         clen_p, int(frag_len), _lib.MEM_HOST, C.byref(h)))
            else:
                chrom = np.ascontiguousarray(gr.seqnames, dtype=np.int32)
                _lib_check(_lib.lib.rcp_reads_load_width(len(gr), _ptr(chrom), 0, None, None, _ptr(start),
                                                         int(fixed), _ptr(strand), clen.shape[0], clen_p,
                                                         int(frag_len), _lib.MEM_HOST, C.byref(h)))
            self.handle = h.value
            self.n = len(gr)
            self.seqlevels = list(gr.seqlevels)
            self._fin = weakref.finalize(self, _free_reads, self.handle)
            return
        end = np.ascontiguousarray(gr.end, dtype=np.int32)
        if use_runs:
            # seqnames held as runs: only the runs cross PCIe
            run_chrom = np.ascontiguousarray(rle.values, dtype=np.int32)
            run_len = np.ascontiguousarray(rle.lengths, dtype=np.int32)
            _lib_check(_lib.lib.rcp_reads_load_rle(len(gr), rle.nrun, _ptr(run_chrom), _ptr(run_len),
                                                   _ptr(start), _ptr(end), _ptr(strand), clen.shape[0],
                                                   clen_p, int(frag_len), _lib.MEM_HOST, C.byref(h)))
        else:
            chrom = np.ascontiguousarray(gr.seqnames, dtype=np.int32)
            _lib_check(_lib.lib.rcp_reads_load(len(gr), _ptr(chrom), _ptr(start), _ptr(end),
                                               _ptr(strand), clen.shape[0], clen_p, int(frag_len),
                                               _lib.MEM_HOST, C.byref(h)))
        self.handle = h.value
        self.n = len(gr)
        self.seqlevels = list(gr.seqlevels)
        self._fin = weakref.finalize(self, _free_reads, self.handle)

    def free(self):
        self._fin()


def _free_reads(h):
    try:
        _lib.lib.rcp_reads_free(h)
    except Exception:
        pass


def _free_cov(h):
    try:
        _lib.lib.rcp_coverage_free(h)
    except Exception:
        pass


def device_reads(gr, frag_len=0):
    """Upload (once) and return the device index of a reads GRanges."""
    key = int(frag_len)
    dr = gr._device.get(key)
    if dr is None:
        dr = DeviceReads(gr, key)
        gr._device[key] = dr
    return dr


class CoverageList:
    """The `$coverage` of one sample: named list, one integer vector (5'->3') or None per region,
    kept on the device (contract T1, SURVEY 8a).  Indexing copies a region to the host."""

    def __init__(self, handle, names=None):
        self.handle = handle
        self.names = names
        n = C.c_int64(0)
        tot = C.c_int64(0)
        nn = C.c_int64(0)
        sc = C.c_double(1.0)
        _lib_check(_lib.lib.rcp_coverage_info(handle, C.byref(n), C.byref(tot), C.byref(nn),
                                              C.byref(sc)))
        self.n = n.value
        self.total_len = tot.value
        self.n_null = nn.value
        vt = C.c_int(0)
        _lib_check(_lib.lib.rcp_coverage_value_type(handle, C.byref(vt)))
        # int32 read counts, or float32 track values (BigWig input)
        self.dtype = np.dtype(np.float32) if vt.value == _lib.VALUE_FLOAT32 else np.dtype(np.int32)
        self._lengths = None
        self._fin = weakref.finalize(self, _free_cov, handle)

    def __len__(self):
        return self.n

    @property
    def scale(self):
        sc = C.c_double(1.0)
        _lib_check(_lib.lib.rcp_coverage_info(self.handle, None, None, None, C.byref(sc)))
        return sc.value

    def set_scale(self, factor):
        """Linear normalisation (recoup.R:559-577): coverage * factor."""
        _lib_check(_lib.lib.rcp_coverage_set_scale(self.handle, float(factor)))

    def lengths(self):
        """`lengths(coverage)`: 0 for NULL entries (profile.R:6)."""
        if self._lengths is None:
            out = np.zeros(self.n, dtype=np.int32)
            _lib_check(_lib.lib.rcp_coverage_lengths(self.handle,
                                                     out.ctypes.data_as(C.POINTER(C.c_int32))))
            self._lengths = out
        return self._lengths

    def is_null(self):
        return self.lengths() == 0

    def fetch(self, first=0, count=None):
        """Unscaled coverage of regions [first, first+count) as a list (None = NULL), of `dtype`."""
        if count is None:
            count = self.n - first
        lens = self.lengths()[first:first + count].astype(np.int64)
        total = int(lens.sum())
        buf = np.zeros(max(total, 1), dtype=self.dtype)
        if self.dtype == np.float32:
            _lib_check(_lib.lib.rcp_coverage_fetch_f32(self.handle, first, count, buf.ctypes.data_as(C.c_void_p),
                                                       total))
        else:
            _lib_check(_lib.lib.rcp_coverage_fetch(self.handle, first, count,
                                                   buf.ctypes.data_as(C.POINTER(C.c_int32)), total))
        out, pos = [], 0
        for l in lens:
            l = int(l)
            out.append(buf[pos:pos + l].copy() if l > 0 else None)
            pos += l
        return out

    def rle(self, first=0, count=None):
        """Regions [first, first+count) as run-length encodings, the `Rle` objects calcCoverage
        returns in the reference (coverage.R:171-173): a list of (values, lengths) array pairs
        (values of `dtype`, lengths int32), None for NULL.  Encoded on the device; only the runs
        are copied."""
        if count is None:
            count = self.n - first
        f32 = self.dtype == np.float32
        rle = _lib.lib.rcp_coverage_rle_f32 if f32 else _lib.lib.rcp_coverage_rle
        ptr = np.zeros(count + 1, dtype=np.int64)
        pp = ptr.ctypes.data_as(C.POINTER(C.c_int64))
        _lib_check(rle(self.handle, first, count, pp, None, None, 0))
        total = int(ptr[count])
        vals = np.zeros(max(total, 1), dtype=self.dtype)
        lens = np.zeros(max(total, 1), dtype=np.int32)
        i32 = C.POINTER(C.c_int32)
        _lib_check(rle(self.handle, first, count, pp, vals.ctypes.data if f32 else vals.ctypes.data_as(i32),
                       lens.ctypes.data_as(i32), total))
        null = self.is_null()[first:first + count]
        return [None if null[i] else (vals[ptr[i]:ptr[i + 1]].copy(), lens[ptr[i]:ptr[i + 1]].copy())
                for i in range(count)]

    def __getitem__(self, i):
        if isinstance(i, str):
            i = self.names.index(i)
        if i < 0:
            i += self.n
        return self.fetch(i, 1)[0]

    def to_list(self):
        return self.fetch(0, self.n)

    def free(self):
        self._fin()


# ------------------------------------------------------------------------------------------------
# calcCoverage
# ------------------------------------------------------------------------------------------------
def _as_reads(input):
    if isinstance(input, GRanges):
        return input
    if isinstance(input, dict) or (isinstance(input, (list, tuple)) and input
                                   and all(isinstance(x, GRanges) for x in input)):
        parts = list(input.values()) if isinstance(input, dict) else list(input)
        first = parts[0]
        cat = GRanges(np.concatenate([p.seqnames for p in parts]),
                      np.concatenate([p.start for p in parts]),
                      np.concatenate([p.end for p in parts]),
                      strand=np.concatenate([p.strand for p in parts]),
                      seqlevels=first.seqlevels, seqlengths=first.seqlengths)
        return cat
    return None


def _map_chrom(mask_gr, reads_gr):
    """Region chromosome ids in the READS' seqlevels; -1 when the chromosome is unknown there
    (coverage.R:189,194-197: 'not found' -> NULL)."""
    if mask_gr.seqlevels == reads_gr.seqlevels:
        return mask_gr.seqnames
    lut = {s: i for i, s in enumerate(reads_gr.seqlevels)}
    table = np.array([lut.get(s, -1) for s in mask_gr.seqlevels], dtype=np.int32)
    return table[mask_gr.seqnames]


_BIGWIG_PATH = re.compile(r"\.(bigwig|bw)$", re.IGNORECASE)     # the reference's dispatch
_BAD_INPUT = ("The input argument must be a GenomicRanges object or a valid "
              "BAM/BigWig file or a list of GenomicRanges")                        # coverage.R:129


def _signal_coverage(track, mask):
    """rcp_signal_coverage of a BigWigTrack over a GRanges / GRangesList mask."""
    h = C.c_int(0)
    gr = mask.unlisted if isinstance(mask, GRangesList) else mask
    chrom = np.ascontiguousarray(_map_chrom(gr, track), dtype=np.int32)     # -1: not in the track
    start = np.ascontiguousarray(gr.start, dtype=np.int32)
    end = np.ascontiguousarray(gr.end, dtype=np.int32)
    strand = np.ascontiguousarray(gr.strand, dtype=np.int8)
    ptr = None
    if isinstance(mask, GRangesList):
        ptr = np.ascontiguousarray(mask.ptr, dtype=np.int64).ctypes.data_as(C.POINTER(C.c_int64))
    _lib_check(_lib.lib.rcp_signal_coverage(track.handle, len(mask), ptr, _ptr(chrom), _ptr(start), _ptr(end),
                                            _ptr(strand), _lib.MEM_HOST, C.byref(h)))
    return CoverageList(h.value, names=mask.names)


def calcCoverage(input, mask, strand=None, ignore_strand=True, rc=None, frag_len=0):
    """coverage.R:126-174.  Returns a CoverageList named by names(mask).  `input` may also be a
    BigWigTrack or a path ending in .bigwig / .bw (coverageFromBigWig, coverage.R:228-322): the
    coverage then holds the track's float32 values, and `strand` / `ignore_strand` have nothing to
    act on (a bigWig has no strand)."""
    from .readers import BigWigTrack, readBigWig
    track, owned = None, False
    if isinstance(input, BigWigTrack):
        track = input
    elif isinstance(input, str) and _BIGWIG_PATH.search(input):
        if not os.path.isfile(input):
            raise ValueError(_BAD_INPUT)
        track, owned = readBigWig(input), True
    reads = None if track is not None else _as_reads(input)
    if reads is None and track is None:
        if isinstance(input, str):
            raise NotImplementedError("BAM file input (coverage.R:228-322) is file I/O, "
                                      "outside the accelerated path; pass decoded ranges")
        raise ValueError(_BAD_INPUT)
    if not isinstance(mask, (GRanges, GRangesList)):
        raise ValueError("The mask argument must be a GRanges or GRangesList object")  # coverage.R:132
    if track is not None:
        try:
            return _signal_coverage(track, mask)
        finally:
            if owned:
                track.free()
    if strand is not None:
        _message("Retrieving ", strand, " reads...")                                    # coverage.R:142
        strand_filter = int(strand_to_code(strand)[0])
    else:
        strand_filter = _lib.STRAND_ANY
    dr = device_reads(reads, frag_len)
    h = C.c_int(0)
    if isinstance(mask, GRangesList):
        u = mask.unlisted
        chrom = np.ascontiguousarray(_map_chrom(u, reads), dtype=np.int32)
        start = np.ascontiguousarray(u.start, dtype=np.int32).copy()
        end = np.ascontiguousarray(u.end, dtype=np.int32).copy()
        bad = chrom < 0
        if bad.any():      # unknown chromosome: make every such range unsatisfiable
            chrom = np.where(bad, 0, chrom).astype(np.int32)
            start[bad] = -1
            end[bad] = -1
        ptr = np.ascontiguousarray(mask.ptr, dtype=np.int64)
        _lib_check(_lib.lib.rcp_coverage_list(dr.handle, len(mask),
                                              ptr.ctypes.data_as(C.POINTER(C.c_int64)), _ptr(chrom),
                                              _ptr(start), _ptr(end), _ptr(u.strand),
                                              int(bool(ignore_strand)), strand_filter,
                                              _lib.MEM_HOST, C.byref(h)))
    else:
        chrom = np.ascontiguousarray(_map_chrom(mask, reads), dtype=np.int32)
        start = np.ascontiguousarray(mask.start, dtype=np.int32)
        end = np.ascontiguousarray(mask.end, dtype=np.int32)
        bad = chrom < 0
        if bad.any():
            chrom = np.where(bad, 0, chrom).astype(np.int32)
            start = np.where(bad, -1, start).astype(np.int32)
            end = np.where(bad, -1, end).astype(np.int32)
        _lib_check(_lib.lib.rcp_coverage(dr.handle, len(mask), _ptr(chrom), _ptr(start), _ptr(end),
                                         _ptr(mask.strand), int(bool(ignore_strand)), strand_filter,
                                         _lib.MEM_HOST, C.byref(h)))
    return CoverageList(h.value, names=mask.names)


def _concat3(left, center, right, names):
    h = C.c_int(0)
    _lib_check(_lib.lib.rcp_coverage_concat3(left.handle, center.handle, right.handle, C.byref(h)))
    return CoverageList(h.value, names=names)


# ------------------------------------------------------------------------------------------------
# coverageRef / coverageRnaRef
# ------------------------------------------------------------------------------------------------
def _stranded(strandedParams):
    sp = strandedParams or {}
    return sp.get("strand"), sp.get("ignoreStrand", True)


def coverageRef(input, genomeRanges, region="tss", flank=(2000, 2000), strandedParams=None,
                bamParams=None, rc=None):
    """coverage.R:1-77.  `input` is the list of sample dicts (id, name, ranges, ...); samples
    whose `coverage` is already set are recomputed only if some sample lacks it (coverage.R:4-6)."""
    if isinstance(region, (list, tuple)):
        region = region[0]
    if all(x.get("coverage") is not None for x in input):
        return input
    strand, ignore = _stranded(strandedParams)
    mainRanges = getRegionalRanges(genomeRanges, region, flank)            # coverage.R:28,46
    for x in input:
        _message("Calculating ", region, " coverage for ", x.get("name"))
        track = _sample_track(x)
        if track is not None:
            x["coverage"] = calcCoverage(track, mainRanges)
            track.free()
            continue
        x["coverage"] = calcCoverage(x["ranges"], mainRanges, strand=strand, ignore_strand=ignore,
                                     rc=rc)
    return input


def _sample_track(x):
    """The BigWigTrack of a sample without reads whose format is "bigwig" (readRanges gives it
    no ranges; the coverage comes from the file).  None for a sample with ranges; any other
    sample without ranges is outside the accelerated path."""
    if x.get("ranges") is not None:
        return None
    if x.get("format") == "bigwig" and x.get("file") is not None:
        from .readers import readBigWig
        return readBigWig(x["file"])
    raise NotImplementedError("sample %r has no decoded ranges; BAM input is outside the accelerated "
                              "path" % (x.get("id"),))


def coverageRnaRef(input, genomeRanges, helperRanges, flank, strandedParams=None, bamParams=None,
                   rc=None):
    """coverage.R:79-124: exon coverage stitched per gene plus the two flanks, NULL if any part is
    NULL.  Keeps the reference's quirk of testing flank[1] for BOTH sides (coverage.R:84-91)."""
    if all(x.get("coverage") is not None for x in input):
        return input
    strand, ignore = _stranded(strandedParams)
    f1, f2 = int(flank[0]), int(flank[1])
    leftRanges = getFlankingRanges(helperRanges, 1 if f1 == 0 else f1, "upstream")
    rightRanges = getFlankingRanges(helperRanges, 1 if f1 == 0 else f2, "downstream")
    for x in input:
        track = _sample_track(x)            # one load serves the three passes
        src = x["ranges"] if track is None else track
        _message("Calculating genebody coverage for ", x.get("name"))
        center = calcCoverage(src, genomeRanges, strand=strand, ignore_strand=ignore, rc=rc)
        left = calcCoverage(src, leftRanges, strand=strand, ignore_strand=ignore, rc=rc)
        right = calcCoverage(src, rightRanges, strand=strand, ignore_strand=ignore, rc=rc)
        x["coverage"] = _concat3(left, center, right, genomeRanges.names)   # coverage.R:115-121
        left.free()
        center.free()
        right.free()
        if track is not None:
            track.free()
    return input
