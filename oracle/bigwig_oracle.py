"""BigWig input of calcCoverage (coverageFromBigWig, R/coverage.R:228-322), restated in plain numpy.

PARITY UNPINNED: the reference cannot run here and its BigWig lines are not part of this
repository, so these are the documented semantics of rtracklayer's import.bw(file, as =
"RleList") and of R subscripting, as recorded in DESIGN.md section 2:

  * import.bw(..., as = "RleList")[[chr]] is a numeric vector of length seqlengths(chr): the value
    of the item that covers a position, 0 where no item does;
  * one element (a GRanges range, or the ranges of one GRangesList element) takes its chromosome
    and strand from its FIRST range (coverage.R:182,185); the index vector is the concatenation
    of start:end over its ranges and follows the same subscript rules as the reads path
    (recoup_oracle._index_subscript): an index past chromSize or a negative index -> NULL, a 0 is
    dropped; the vector is reversed on '-';
  * NULL also when the chromosome is not in the track or no index is left; a window that no item
    overlaps is a zero vector, NOT NULL (unlike the reads path, where zero reads mean NULL);
  * values are float32; NaN / Inf are refused by the loader; -0.0 reads as +0.0.

Items are (chrom, start, end, value) with 1-based closed coordinates.
"""
import numpy as np

from .recoup_oracle import _index_subscript


class Track:
    def __init__(self, chrom, start, end, value, chrom_sizes):
        self.chrom = np.asarray(chrom, dtype=np.int64)
        self.start = np.asarray(start, dtype=np.int64)
        self.end = np.asarray(end, dtype=np.int64)
        self.value = np.asarray(value, dtype=np.float32)
        if np.any(np.diff(self.chrom) < 0) or np.any((np.diff(self.start) < 0) & (np.diff(self.chrom) == 0)):
            order = np.lexsort((self.start, self.chrom))
            self.chrom, self.start, self.end, self.value = (x[order] for x in
                                                            (self.chrom, self.start, self.end, self.value))
        self.value = np.where(self.value == 0, np.float32(0), self.value).astype(np.float32)
        self.chrom_sizes = np.asarray(chrom_sizes, dtype=np.int64)
        self.ptr = np.searchsorted(self.chrom, np.arange(self.chrom_sizes.shape[0] + 1))

    @classmethod
    def from_file_items(cls, items, chrom_sizes):
        """items: (chrom, start0, end0, value) as stored in the file (0-based half-open)."""
        a = np.asarray([(c, s + 1, e) for c, s, e, _ in items], dtype=np.int64).reshape(-1, 3)
        v = np.asarray([x[3] for x in items], dtype=np.float32)
        return cls(a[:, 0], a[:, 1], a[:, 2], v, chrom_sizes)

    def chrom_vector(self, c):
        """The whole numeric vector of chromosome c (positions 1..chromSize)."""
        out = np.zeros(int(self.chrom_sizes[c]), dtype=np.float32)
        a, b = self.ptr[c], self.ptr[c + 1]
        for s, e, v in zip(self.start[a:b], self.end[a:b], self.value[a:b]):
            out[s - 1:e] = v
        return out

    def values_at(self, c, idx):
        """chrom_vector(c)[idx - 1] without building the vector (idx 1-based, in bounds)."""
        a, b = self.ptr[c], self.ptr[c + 1]
        s, e, v = self.start[a:b], self.end[a:b], self.value[a:b]
        out = np.zeros(idx.shape[0], dtype=np.float32)
        if s.size == 0:
            return out
        k = np.searchsorted(s, idx, side="right") - 1         # last item starting at or before idx
        ok = (k >= 0) & (idx <= e[np.clip(k, 0, None)])
        out[ok] = v[k[ok]]
        return out


def coverage_from_track(track, chrom, starts, ends, strands):
    """One element: float32 vector or None."""
    starts = np.atleast_1d(np.asarray(starts, dtype=np.int64))
    ends = np.atleast_1d(np.asarray(ends, dtype=np.int64))
    strands = np.atleast_1d(np.asarray(strands, dtype=np.int64))
    if starts.size == 0 or chrom < 0 or chrom >= track.chrom_sizes.shape[0]:
        return None
    idx = np.concatenate([np.arange(s, e + 1, dtype=np.int64) for s, e in zip(starts, ends)])
    idx = _index_subscript(int(track.chrom_sizes[chrom]), idx)
    if idx is None or idx.size == 0:
        return None
    out = track.values_at(chrom, idx)
    if int(strands[0]) < 0:
        out = out[::-1]
    return np.ascontiguousarray(out)


def calc_coverage(track, mask):
    """calcCoverage(<bigwig>, mask): `mask` as in recoup_oracle.calc_coverage, chromosome ids in
    the track's chromosomes (-1: not in the track)."""
    chrom = np.asarray(mask["chrom"], dtype=np.int64)
    ms = np.asarray(mask["start"], dtype=np.int64)
    me = np.asarray(mask["end"], dtype=np.int64)
    mst = np.asarray(mask["strand"], dtype=np.int64)
    out = []
    if "ptr" in mask:
        ptr = np.asarray(mask["ptr"], dtype=np.int64)
        for i in range(ptr.shape[0] - 1):
            a, b = int(ptr[i]), int(ptr[i + 1])
            out.append(None if b <= a else coverage_from_track(track, int(chrom[a]), ms[a:b], me[a:b], mst[a:b]))
    else:
        for i in range(ms.shape[0]):
            out.append(coverage_from_track(track, int(chrom[i]), ms[i:i + 1], me[i:i + 1], mst[i:i + 1]))
    return out
