"""Host mirror of the read-import step right before the hot path, for reads that are already
decoded (SURVEY 8f N3):

    preprocessRanges(input, preprocessParams, bamParams, rc)            ranges.R:1-65
    readBam(..., sa = "remove", sq)                                     ranges.R:125-133

The decode itself: `reader`, a callable that returns the decoded GRanges of one sample (what
readBam / readBed would return for spliceAction "keep" or "split"), or -- reader None -- the
sample's own `file` / `format` through the device decoders of readers.py (BAM records and BED text
parsed on the device after the host's BGZF inflate).  Everything after the decode runs here: the width cut of spliceAction "remove" (a type-7 quantile, on the device), the seeded
down-sampling indices (base R's sample() stream, serial by nature: host code inside the library)
and the selection itself, which the device applies while it loads the reads
(rcp_reads_load_select) -- the selected reads are never gathered on the host unless somebody
reads their coordinates.
"""
import ctypes as C

import numpy as np

from . import _lib
from .coverage import _message
from .ranges import GRanges


class SelectedGRanges(GRanges):
    """`parent[-which(width(parent) > max_width)][idx]` kept as (parent, selection)."""

    def __init__(self, parent, n_kept, max_width=None, idx=None):
        self.parent = parent
        self.max_width = max_width
        self.idx = None if idx is None else np.ascontiguousarray(idx, dtype=np.int32)
        self._n = int(n_kept) if idx is None else int(self.idx.shape[0])
        self.seqlevels = list(parent.seqlevels)
        self.seqlengths = parent.seqlengths
        self.names = None
        self.seqnames_rle = None
        self.fixed_width = None
        self._device = {}
        self._host = None

    def __len__(self):
        return self._n

    def _materialise(self):
        if self._host is None:
            p = self.parent
            pos = np.arange(len(p))
            if self.max_width is not None:
                pos = pos[~(p.width > self.max_width)]
            if self.idx is not None:
                pos = pos[self.idx.astype(np.int64) - 1]
            self._host = (p.seqnames[pos], p.start[pos], p.end[pos], p.strand[pos])
        return self._host

    seqnames = property(lambda self: self._materialise()[0])
    start = property(lambda self: self._materialise()[1])
    end = property(lambda self: self._materialise()[2])
    strand = property(lambda self: self._materialise()[3])


def widthQuantile(gr, prob):
    """(quantile(width(gr), prob), number of reads not wider than it)"""
    _lib.ensure_init()
    if getattr(gr, "decoded_handle", None) is not None:      # decoded on the device: stays there
        q, n_le = C.c_double(0.0), C.c_int64(0)
        _lib.check(_lib.lib.rcp_decoded_width_quantile(gr.decoded_handle, float(prob), C.byref(q), C.byref(n_le)))
        return q.value, n_le.value
    start = np.ascontiguousarray(gr.start, dtype=np.int32)
    end = np.ascontiguousarray(gr.end, dtype=np.int32)
    q = C.c_double(0.0)
    n_le = C.c_int64(0)
    _lib.check(_lib.lib.rcp_reads_width_quantile(len(gr), start.ctypes.data_as(C.c_void_p),
                                                 end.ctypes.data_as(C.c_void_p), float(prob),
                                                 _lib.MEM_HOST, C.byref(q), C.byref(n_le)))
    return q.value, n_le.value


def sampleSorted(lib_sizes, size, seed, sample_kind="Rejection"):
    """set.seed(seed); lapply(libSizes, function(x, s) sort(sample(x, s)), size)"""
    n = np.ascontiguousarray(lib_sizes, dtype=np.int64)
    k = np.full(n.shape[0], int(size), dtype=np.int64)
    out = np.empty(int(k.sum()), dtype=np.int32)
    i64 = C.POINTER(C.c_int64)
    _lib.check(_lib.lib.rcp_r_sample_sorted(int(seed), _lib.SAMPLE_KIND[sample_kind], n.shape[0],
                                            n.ctypes.data_as(i64), k.ctypes.data_as(i64),
                                            out.ctypes.data_as(C.c_void_p)))
    return [out[i * int(size):(i + 1) * int(size)] for i in range(n.shape[0])]


def readRanges(x, reader, spliceAction="keep", spliceRemoveQ=0.75, bamParams=None):
    """readRanges / readBam after the decode (ranges.R:102-134): "keep" and "split" differ only in
    how the file is decoded (the reader's business); "remove" drops the reads wider than the
    spliceRemoveQ quantile of the widths.  `bamParams` (a ScanBamParam) filters the records of a
    BAM file; BED files and a `reader` callable do not see it."""
    if spliceAction not in ("keep", "remove", "split"):
        raise ValueError("sa must be one of keep, remove, split")
    if not 0 <= spliceRemoveQ <= 1:
        raise ValueError("sq must be in [0, 1]")
    if reader is None:
        # the file itself: decoded on the device (readers.py); "split" is the decoder's business
        from .readers import readRangesFile
        if x.get("file") is None or x.get("format") is None:
            raise ValueError("One or more input files cannot be read: no file / format and no reader")
        gr = readRangesFile(x["file"], x["format"], "split" if spliceAction == "split" else "keep",
                            seqlevels=x.get("seqlevels"), seqlengths=x.get("seqlengths"), bamParams=bamParams)
    else:
        gr = reader(x)
    if spliceAction != "remove" or len(gr) == 0:
        return gr
    qu, n_kept = widthQuantile(gr, spliceRemoveQ)
    _message("  Excluded ", len(gr) - n_kept, " reads")
    return SelectedGRanges(gr, n_kept, max_width=qu)


def preprocessRanges(input, preprocessParams, bamParams=None, rc=None, reader=None,
                     sample_kind="Rejection"):
    """ranges.R:1-65.  Returns `input` untouched when every sample already has `ranges`
    (ranges.R:2-4); else reads ALL samples through `reader` and applies
    preprocessParams$normalize: "none" / "linear" keep the reads as read (linear acts after the
    coverage), "downsample" draws min(library sizes) reads from every sample, "sampleto" draws
    preprocessParams$sampleTo, both with ONE set.seed(preprocessParams$seed).  `bamParams`: a
    ScanBamParam for the BAM files read here (ranges.R:18-19); the library sizes that
    "downsample" / "sampleto" draw from are those of the filtered reads."""
    if not any(x.get("ranges") is None for x in input):
        return input
    pp = preprocessParams
    normalize = pp.get("normalize", "none")
    if normalize not in ("none", "linear", "downsample", "sampleto"):
        raise ValueError("normalize must be one of none, linear, downsample, sampleto")
    ranges = []
    for x in input:
        _message("Reading sample ", x.get("name"))
        ranges.append(readRanges(x, reader, pp.get("spliceAction", "keep"), pp.get("spliceRemoveQ", 0.75),
                                 bamParams))
    if normalize in ("downsample", "sampleto"):
        lib = [len(r) for r in ranges]
        size = min(lib) if normalize == "downsample" else int(pp["sampleTo"])
        idx = sampleSorted(lib, size, pp.get("seed", 42), sample_kind)
        out = []
        for r, ix in zip(ranges, idx):
            if isinstance(r, SelectedGRanges):
                out.append(SelectedGRanges(r.parent, len(r), max_width=r.max_width, idx=ix))
            else:
                out.append(SelectedGRanges(r, len(r), idx=ix))
        ranges = out
    for x, r in zip(input, ranges):
        x["ranges"] = r
    return input
