"""Host mirror of the reference's file readers (ranges.R:102-146) over the device decoders
(SURVEY 8f N3):

    readBam(bam, sa = c("keep", "remove", "split"), sq = 0.75)        ranges.R:111-134
    readBed(bed, bg)                                                  ranges.R:136-146
    readBigWig(bw)                  import.bw(bw) of coverageFromBigWig, coverage.R:228-322

What stays on the host: opening the file, the BGZF inflate (rcp_bgzf_inflate: zlib, one thread per
core, C++ inside the library), the BAM header (text + reference list) and the walk of the
length-prefixed record chain (rcp_bam_index, also inside the library).  Everything per read -- flag
filter and the other ScanBamParam filters, CIGAR walk, N-split, trim, text parsing, compaction in file
order (or in `which` order) -- runs on the device (rcp_bam_decode[_param] / rcp_bed_decode); the decoded reads stay in
HBM and go to the hot path without a host round trip (rcp_reads_load_decoded).  Their coordinates
are copied to the host only when somebody reads them.  A bigWig track is parsed and inflated on the
host (rcp_bigwig_load, threads inside the library) and expanded into items on the device; its items
stay in HBM behind a `signal` handle.
"""
import ctypes as C
import gzip
import struct
import weakref

import numpy as np

from . import _lib
from .coverage import _message
from .preprocess import SelectedGRanges, widthQuantile
from .ranges import GRanges


def _free_decoded(h):
    try:
        _lib.lib.rcp_decoded_free(h)
    except Exception:
        pass


class DecodedGRanges(GRanges):
    """The reads of one file, decoded on the device (a `decoded` handle)."""

    def __init__(self, handle, n, seqlevels, seqlengths):
        self.decoded_handle = int(handle)
        self._n = int(n)
        self.seqlevels = list(seqlevels)
        self.seqlengths = None if seqlengths is None else np.ascontiguousarray(seqlengths, dtype=np.int64)
        self.names = None
        self.seqnames_rle = None
        self.fixed_width = None
        self._device = {}
        self._host = None
        self._fin = weakref.finalize(self, _free_decoded, self.decoded_handle)

    def __len__(self):
        return self._n

    def _materialise(self):
        if self._host is None:
            n = self._n
            chrom, start, end = (np.zeros(n, dtype=np.int32) for _ in range(3))
            strand = np.zeros(n, dtype=np.int8)
            p = lambda a: a.ctypes.data_as(C.c_void_p)
            _lib.check(_lib.lib.rcp_decoded_fetch(self.decoded_handle, p(chrom), p(start), p(end), p(strand), n))
            self._host = (chrom, start, end, strand)
        return self._host

    seqnames = property(lambda self: self._materialise()[0])
    start = property(lambda self: self._materialise()[1])
    end = property(lambda self: self._materialise()[2])
    strand = property(lambda self: self._materialise()[3])

    @property
    def width(self):
        return self.end.astype(np.int64) - self.start.astype(np.int64) + 1


def bgzfInflate(data, threads=0):
    """The inflated bytes of a BGZF file as a uint8 array: the library's multi-threaded inflate
    (rcp_bgzf_inflate), or python's gzip for data that is gzip but not BGZF."""
    buf = np.frombuffer(bytes(data) if not isinstance(data, (bytes, bytearray)) else data, dtype=np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    total, nblk = C.c_int64(0), C.c_int64(0)
    if _lib.lib.rcp_bgzf_size(vp(buf), buf.shape[0], C.byref(total), C.byref(nblk)) != _lib.RCP_OK:
        return np.frombuffer(gzip.decompress(bytes(data)), dtype=np.uint8)
    out = np.empty(total.value, dtype=np.uint8)
    _lib.check(_lib.lib.rcp_bgzf_inflate(vp(buf), buf.shape[0], vp(out), out.shape[0], int(threads)))
    return out


def bam_header(raw):
    """(seqlevels, seqlengths, offset of the first alignment record) of an inflated BAM."""
    raw = memoryview(raw)
    if bytes(raw[:4]) != b"BAM\x01":
        raise ValueError("not a BAM file (magic %r)" % bytes(raw[:4]))
    l_text, = struct.unpack_from("<i", raw, 4)
    p = 8 + l_text
    n_ref, = struct.unpack_from("<i", raw, p)
    p += 4
    names, lens = [], []
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", raw, p)
        names.append(bytes(raw[p + 4:p + 4 + l_name - 1]).decode("ascii"))
        ln, = struct.unpack_from("<i", raw, p + 4 + l_name)
        lens.append(ln)
        p += 8 + l_name
    return names, np.asarray(lens, dtype=np.int64), p


FLAG_BITS = ("isPaired", "isProperPair", "isUnmappedQuery", "hasUnmappedMate", "isMinusStrand",
             "isMateMinusStrand", "isFirstMateRead", "isSecondMateRead", "isSecondaryAlignment",
             "isNotPassingQualityControls", "isDuplicate", "isSupplementaryAlignment")   # 0x1 .. 0x800
WHICH_MAX_END = 536870912       # 2^29, the largest end Rsamtools accepts


def scanBamFlag(isPaired=None, isProperPair=None, isUnmappedQuery=None, hasUnmappedMate=None,
                isMinusStrand=None, isMateMinusStrand=None, isFirstMateRead=None, isSecondMateRead=None,
                isSecondaryAlignment=None, isNotPassingQualityControls=None, isDuplicate=None,
                isSupplementaryAlignment=None):
    """Rsamtools' scanBamFlag: each argument True, False or None (NA).  Returns the pair
    bamFlag(asInteger = TRUE) = (keep0, keep1): True clears the bit in keep0 (only records with
    the bit set pass), False clears it in keep1 (only records with it clear pass)."""
    args = locals()
    keep0 = keep1 = 0xfff
    for bit, name in enumerate(FLAG_BITS):
        v = args[name]
        if v is None:
            continue
        if not isinstance(v, (bool, np.bool_)):
            raise ValueError("scanBamFlag: %s must be True, False or None" % name)
        if v:
            keep0 &= ~(1 << bit)
        else:
            keep1 &= ~(1 << bit)
    return keep0, keep1


class ScanBamParam:
    """Rsamtools' ScanBamParam, the parts that decide which alignments readGAlignments returns:

    flag         a (keep0, keep1) pair from scanBamFlag; None = every record (unmapped records are
                 dropped whatever it says: readGAlignments ANDs isUnmappedQuery = FALSE in).
    mapqFilter   keep MAPQ >= mapqFilter; None = NA, no filter.
    which        a GRanges, or a list of (seqname, start, end), 1-based closed.  The output is
                 range by range in the order of as(which, "IntegerRangesList") -- grouped by the
                 seqlevels of `which` in level order (for a list: the order the seqnames first
                 appear in), ranges in their given order within a level, file order within a
                 range -- and a record overlapping k ranges is returned k times.  Needs the
                 records sorted by position.
    simpleCigar  keep only alignments whose CIGAR is one M operation.
    tagFilter    {tag: accepted values}: a record passes iff every tag is present with one of
                 its values; integers match integer fields, strings Z and A fields.
    what, tag, reverseComplement  accepted; they only touch columns that as(., "GRanges") drops.
    """

    def __init__(self, flag=None, mapqFilter=None, which=None, simpleCigar=False, tagFilter=None,
                 what=None, tag=None, reverseComplement=False):
        if flag is None:
            flag = (0xfff, 0xfff)
        if (len(flag) != 2 or any(isinstance(x, bool) or int(x) != x or not 0 <= int(x) <= 0xfff for x in flag)):
            raise ValueError("flag must be a (keep0, keep1) pair of 12-bit masks, as scanBamFlag returns")
        self.flag = (int(flag[0]), int(flag[1]))
        if mapqFilter is not None:
            if isinstance(mapqFilter, bool) or int(mapqFilter) != mapqFilter or mapqFilter < 0:
                raise ValueError("mapqFilter must be a non-negative integer or None")
            mapqFilter = int(mapqFilter)
        self.mapqFilter = mapqFilter
        if not isinstance(simpleCigar, (bool, np.bool_)):
            raise ValueError("simpleCigar must be True or False")
        self.simpleCigar = bool(simpleCigar)
        self.which = None if which is None else _which_ranges(which)
        if self.which is not None:      # the same as arrays: level names, level index, start, end
            levels = list(dict.fromkeys(c for c, _, _ in self.which))
            lut = {c: i for i, c in enumerate(levels)}
            self._which_arrays = (levels, np.asarray([lut[c] for c, _, _ in self.which], dtype=np.int32),
                                  np.asarray([x[1] for x in self.which], dtype=np.int32),
                                  np.asarray([x[2] for x in self.which], dtype=np.int32))
        self.tagFilter = {}
        for name, values in (tagFilter or {}).items():
            if not isinstance(name, str) or len(name) != 2:
                raise ValueError("tagFilter: tag name %r is not 2 characters" % (name,))
            vals = list(values) if isinstance(values, (list, tuple, np.ndarray)) else [values]
            is_str = [isinstance(v, str) for v in vals]
            if any(is_str) and not all(is_str):
                raise ValueError("tagFilter: tag %s mixes integer and character values" % name)
            if not all(is_str) and any(isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer))
                                       for v in vals):
                raise ValueError("tagFilter: tag %s: values must be integers or strings" % name)
            self.tagFilter[name] = [v if isinstance(v, str) else int(v) for v in vals]
        self.what, self.tag, self.reverseComplement = what, tag, reverseComplement

    def keep_words(self):
        """The flag pair readGAlignments applies: the user's AND isUnmappedQuery = FALSE."""
        return self.flag[0], self.flag[1] & ~0x4


def _which_ranges(which):
    """[(seqname, start, end)] in IntegerRangesList order, validated."""
    if isinstance(which, GRanges):
        ids = np.asarray(which.seqnames)
        rows = [(which.seqlevels[int(c)], int(s), int(e)) for c, s, e in zip(ids, which.start, which.end)]
        levels = list(which.seqlevels)
    else:
        rows = [(str(c), int(s), int(e)) for c, s, e in which]
        levels = list(dict.fromkeys(c for c, _, _ in rows))
    for c, s, e in rows:
        if s < 1 or e < s or e > WHICH_MAX_END:
            raise ValueError("which: range %s:%d-%d needs 1 <= start <= end <= %d" % (c, s, e, WHICH_MAX_END))
    rank = {c: i for i, c in enumerate(levels)}
    return sorted(rows, key=lambda x: rank[x[0]])          # stable: the given order within a level


def decodeBam(raw, split=False, params=None):
    """Inflated BAM bytes -> DecodedGRanges: readGAlignments (with `params`, a ScanBamParam) +
    as(., "GRanges") (or unlist(grglist(.)) when `split`) + trim."""
    _lib.ensure_init()
    names, lens, first = bam_header(raw)
    rec = np.frombuffer(raw, dtype=np.uint8, offset=first)
    n_rec = C.c_int64(0)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib.rcp_bam_index(vp(rec), rec.shape[0], C.byref(n_rec), None, 0))
    off = np.zeros(n_rec.value + 1, dtype=np.int64)
    _lib.check(_lib.lib.rcp_bam_index(vp(rec), rec.shape[0], C.byref(n_rec), vp(off), off.shape[0]))
    h, n_out = C.c_int(0), C.c_int64(0)
    lens_p = lens.ctypes.data_as(C.POINTER(C.c_int64))
    if params is None:
        _lib.check(_lib.lib.rcp_bam_decode(vp(rec), rec.shape[0], vp(off), n_rec.value, len(names), lens_p,
                                           1 if split else 0, _lib.MEM_HOST, C.byref(h), C.byref(n_out)))
    else:
        _lib.check(bam_decode_param(vp(rec), rec.shape[0], vp(off), n_rec.value, names, lens, split, _lib.MEM_HOST,
                                    params, h, n_out))
    return DecodedGRanges(h.value, n_out.value, names, lens)


def bam_decode_param(rec, n_bytes, off, n_rec, names, lens, split, mem, params, h, n_out):
    """rcp_bam_decode_param with the arguments of a ScanBamParam; returns the status code."""
    i32p = C.POINTER(C.c_int32)
    a32 = lambda x: np.ascontiguousarray(x, dtype=np.int32)
    flag = a32(params.keep_words())
    n_which, w_ref, w_start, w_end = 0, a32([]), a32([]), a32([])
    if params.which is not None:
        levels, level_idx, w_start, w_end = params._which_arrays
        lut = {c: i for i, c in enumerate(names)}
        for c in levels:
            if c not in lut:
                raise ValueError("which: seqname %s is not among the BAM header's references" % c)
        w_ref = a32([lut[c] for c in levels])[level_idx] if levels else a32([])
        n_which = w_ref.shape[0]
    tags = list(params.tagFilter.items())
    tag_names = "".join(t for t, _ in tags).encode("ascii")
    tag_ptr = a32(np.cumsum([0] + [len(v) for _, v in tags]))
    tag_type = a32([1 if v and isinstance(v[0], str) else 0 for _, v in tags])
    flat = [x for _, v in tags for x in v]
    int_values = np.asarray([x if isinstance(x, int) else 0 for x in flat], dtype=np.int64)
    str_values = (C.c_char_p * max(len(flat), 1))(*[x.encode("utf-8") if isinstance(x, str) else b"" for x in flat])
    lens = np.ascontiguousarray(lens, dtype=np.int64)
    return _lib.lib.rcp_bam_decode_param(
        rec, n_bytes, off, n_rec, len(names), lens.ctypes.data_as(C.POINTER(C.c_int64)), 1 if split else 0, mem,
        flag.ctypes.data_as(i32p), -1 if params.mapqFilter is None else params.mapqFilter,
        1 if params.simpleCigar else 0, n_which, w_ref.ctypes.data_as(i32p), w_start.ctypes.data_as(i32p),
        w_end.ctypes.data_as(i32p), len(tags), tag_names, tag_ptr.ctypes.data_as(i32p), tag_type.ctypes.data_as(i32p),
        int_values.ctypes.data_as(C.POINTER(C.c_int64)), str_values, C.byref(h), C.byref(n_out))


def readBam(bam, sa="keep", sq=0.75, params=None):
    """ranges.R:111-134.  `bam`: a path, or the bytes of the file; `params`: a ScanBamParam (the
    reference's bamParams), None for readGAlignments' default."""
    if sa not in ("keep", "remove", "split"):
        raise ValueError("sa must be one of keep, remove, split")
    if not 0 <= sq <= 1:
        raise ValueError("sq must be in [0, 1]")
    data = bam if isinstance(bam, (bytes, bytearray, memoryview)) else open(bam, "rb").read()
    raw = bgzfInflate(data)                     # BGZF blocks inflated in parallel (host zlib)
    reads = decodeBam(raw, split=(sa == "split"), params=params)
    if sa != "remove" or len(reads) == 0:
        return reads
    qu, n_kept = widthQuantile(reads, sq)
    _message("  Excluded ", len(reads) - n_kept, " reads")
    return SelectedGRanges(reads, n_kept, max_width=qu)


def readBed(bed, seqlevels, seqlengths=None):
    """ranges.R:136-146: import.bed(bed, trackLine = FALSE); the reference then looks the
    chromosome lengths of the genome up (UCSC): here the caller passes them.  `bed`: a path or the
    bytes of the file."""
    _lib.ensure_init()
    data = bed if isinstance(bed, (bytes, bytearray, memoryview)) else open(bed, "rb").read()
    if bytes(data[:2]) == b"\x1f\x8b":
        data = gzip.decompress(bytes(data))
    text = np.frombuffer(bytes(data), dtype=np.uint8)
    arr = (C.c_char_p * len(seqlevels))(*[s.encode("ascii") for s in seqlevels])
    h, n_out = C.c_int(0), C.c_int64(0)
    _lib.check(_lib.lib.rcp_bed_decode(text.ctypes.data_as(C.c_void_p), text.shape[0], len(seqlevels), arr,
                                       _lib.MEM_HOST, C.byref(h), C.byref(n_out)))
    return DecodedGRanges(h.value, n_out.value, seqlevels, seqlengths)


def _free_signal(h):
    try:
        _lib.lib.rcp_signal_free(h)
    except Exception:
        pass


class BigWigTrack:
    """A bigWig track resident on the device (a `signal` handle): its items are the runs of
    import.bw(file, as = "RleList") that are not zero -- start, end (1-based, closed) and a float32
    value.  `seqlevels` / `seqlengths` are the file's chromosomes in chromId order."""

    def __init__(self, handle):
        self.handle = int(handle)
        self._fin = weakref.finalize(self, _free_signal, self.handle)
        n_chrom, n_items, nb = C.c_int(0), C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib.rcp_signal_info(self.handle, C.byref(n_chrom), C.byref(n_items), C.byref(nb)))
        names = C.create_string_buffer(max(nb.value, 1))
        lens = np.zeros(max(n_chrom.value, 1), dtype=np.int64)
        _lib.check(_lib.lib.rcp_signal_chroms(self.handle, names, lens.ctypes.data_as(C.POINTER(C.c_int64))))
        raw = names.raw[:nb.value]
        self.seqlevels = [x.decode("utf-8", "replace") for x in raw.split(b"\0")[:n_chrom.value]]
        self.seqlengths = lens[:n_chrom.value].copy()
        self._n = n_items.value

    def __len__(self):
        return self._n

    def fetch(self):
        """(chrom ids, start, end, value) of every item, in (chromosome, start) order."""
        n = self._n
        chrom, start, end = (np.zeros(max(n, 1), dtype=np.int32) for _ in range(3))
        value = np.zeros(max(n, 1), dtype=np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(_lib.lib.rcp_signal_fetch(self.handle, p(chrom), p(start), p(end), p(value), n))
        return chrom[:n], start[:n], end[:n], value[:n]

    def free(self):
        self._fin()


def readBigWig(bw, threads=0):
    """import.bw(bw) of the whole file (coverage.R:228-322) -> BigWigTrack.  `bw`: a path, or
    the bytes of the file; `threads`: host threads of the inflate (0 = one per core)."""
    _lib.ensure_init()
    data = bw if isinstance(bw, (bytes, bytearray, memoryview)) else open(bw, "rb").read()
    buf = np.frombuffer(bytes(data) if isinstance(data, memoryview) else data, dtype=np.uint8)
    h = C.c_int(0)
    _lib.check(_lib.lib.rcp_bigwig_load(buf.ctypes.data_as(C.c_void_p), buf.shape[0], int(threads), C.byref(h)))
    return BigWigTrack(h.value)


def readRangesFile(input, format, sa="keep", sq=0.75, seqlevels=None, seqlengths=None, bamParams=None):
    """readRanges (ranges.R:102-109) for files; "bigwig" has no reads (NULL: coverageRef reads the
    track itself from the sample's `file`, see readBigWig).  `bamParams` (a
    ScanBamParam) applies to BAM files only, as in the reference."""
    if format == "bam":
        return readBam(input, sa, sq, params=bamParams)
    if format == "bed":
        return readBed(input, seqlevels, seqlengths)
    if format == "bigwig":
        return None
    raise ValueError("format must be one of bam, bed, bigwig")
