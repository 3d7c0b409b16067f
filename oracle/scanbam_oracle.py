"""TEST INFRASTRUCTURE -- CPU restatement of the BAM reader under a ScanBamParam, alongside
oracle/import_oracle.py (the reader without one).  Only tests/ may import this; the product never
does.

`readGAlignments(file, param = ScanBamParam(...))` (the reference's `bamParams`, ranges.R:18-19,
111-134), restated from the Rsamtools / GenomicAlignments man pages (`?ScanBamParam`,
`?scanBamFlag`, `?readGAlignments`) -- **parity unpinned**, like the rest of the import oracle.
`bam_decode(..., params=)` takes a dict with any of these keys; each record is judged on its own,
before the CIGAR walk's ranges are made, and trim() / split / remove act on what passes:

1. `flag` (`?scanBamFlag`, `?ScanBamParam`): the pair `bamFlag(param, asInteger = TRUE)` =
   (keep0, keep1) over the 12 bits isPaired 0x1, isProperPair 0x2, isUnmappedQuery 0x4,
   hasUnmappedMate 0x8, isMinusStrand 0x10, isMateMinusStrand 0x20, isFirstMateRead 0x40,
   isSecondMateRead 0x80, isSecondaryAlignment 0x100, isNotPassingQualityControls 0x200,
   isDuplicate 0x400, isSupplementaryAlignment 0x800.  TRUE clears the bit in keep0, FALSE in keep1,
   NA leaves it in both.  A record passes iff every bit set in FLAG is set in keep1 and every bit
   clear in FLAG is set in keep0.  readGAlignments ANDs `isUnmappedQuery = FALSE` in
   (`bamFlagAND`), so unmapped records stay dropped.
2. `mapqFilter` (`?ScanBamParam`): MAPQ >= mapqFilter; None (NA) = no filter; MAPQ 255 is the
   number 255.
3. `simpleCigar` (`?ScanBamParam`: "only alignments with a 'simple' cigar (e.g. 100M)"): the CIGAR
   is ONE M operation; read here so that 10M5M is not simple.
4. `tagFilter` (`?ScanBamParam`): {tag: accepted values}; a record passes iff every tag is present
   with one of its values.  Integer values match the integer aux types c C s S i I by value,
   character values Z and A fields exactly; a missing tag or one of another type (f, H, B) fails;
   the first occurrence of a tag decides.  The aux fields follow read_name, CIGAR, seq
   ((l_seq+1)/2 bytes) and qual (l_seq bytes) and are walked over every SAMv1 4.2.4 type (B arrays
   of every subtype, NUL-terminated Z / H); a field running past its record is an error.
5. `which` (`?ScanBamParam`: "When one record overlaps two ranges in which, the record is returned
   twice"): (seqname, start, end) ranges, 1-based closed; `which_levels` (default: the seqnames in
   order of first appearance) are the seqlevels of that GRanges.  A record overlaps [s, e] on its
   reference iff pos0 < e and pos0 + rlen > s - 1, rlen = the CIGAR's M D N = X, 1 when that is 0
   (htslib `bam_endpos`), on the file coordinates before trim().  Output order is that of
   `as(which, "IntegerRangesList")`: by level, ranges in their given order within a level, file
   order within a range; a record overlapping k ranges appears k times (each split at its N
   operations under "split").  An index -- hence records sorted by (refID, POS), unplaced ones
   last -- is needed: unsorted records are an error; so are a seqname missing from the header,
   start < 1, end < start and end > 536870912 (the Rsamtools limit).
6. `what`, `tag`, `reverseComplement` only add or alter columns that as(., "GRanges") drops: no
   effect.
"""
import struct

import numpy as np

from .import_oracle import BLOCK_OPS, REF_OPS, _trim


def _ranges_of(ref, pos, ops, L, split):
    """as(., "GRanges") (one range) or grglist() (the blocks between N operations) of one
    alignment, trimmed"""
    if not split:
        w = sum(c >> 4 for c in ops if (c & 15) in REF_OPS)
        return [_trim(pos + 1, pos + w, L)]
    out = []
    cur, blk = pos + 1, 0
    for c in ops:
        op, ln = c & 15, c >> 4
        if op in BLOCK_OPS:
            blk += ln
        elif op == 3:
            if blk > 0:
                out.append(_trim(cur, cur + blk - 1, L))
            cur += blk + ln
            blk = 0
    if blk > 0:
        out.append(_trim(cur, cur + blk - 1, L))
    return out


AUX_SIZE = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}
AUX_INT = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}


def parse_aux(data):
    """The aux fields of one record (SAMv1 4.2.4) -> [(tag, type, value)]; value: int for the
    integer types, str for Z and A, None for the others.  ValueError when a field runs past the end
    or has an unknown type."""
    out, q = [], 0
    while q < len(data):
        if len(data) - q < 3:
            raise ValueError("aux field header runs past the record")
        tag, ty = data[q:q + 2].decode("latin-1"), chr(data[q + 2])
        q += 3
        if ty in AUX_SIZE:
            sz = AUX_SIZE[ty]
        elif ty in "ZH":
            z = data.find(b"\x00", q)
            if z < 0:
                raise ValueError("unterminated %s aux field" % ty)
            sz = z + 1 - q
        elif ty == "B":
            if len(data) - q < 5:
                raise ValueError("B aux field header runs past the record")
            sub = chr(data[q])
            if sub not in "cCsSiIf":
                raise ValueError("B aux field of subtype %r" % sub)
            sz = 5 + struct.unpack_from("<I", data, q + 1)[0] * AUX_SIZE[sub]
        else:
            raise ValueError("aux type %r" % ty)
        if q + sz > len(data):
            raise ValueError("aux field runs past the record")
        if ty in AUX_INT:
            val = struct.unpack_from(AUX_INT[ty], data, q)[0]
        elif ty == "Z":
            val = data[q:q + sz - 1].decode("latin-1")
        elif ty == "A":
            val = chr(data[q])
        else:
            val = None
        out.append((tag, ty, val))
        q += sz
    return out


def _tags_pass(fields, tag_filter):
    first = {}
    for tag, ty, val in fields:
        first.setdefault(tag, (ty, val))
    for tag, values in tag_filter.items():
        if tag not in first:
            return False
        ty, val = first[tag]
        want_str = bool(values) and isinstance(values[0], str)
        if want_str and ty in "ZA":
            ok = val in values
        elif not want_str and ty in AUX_INT:
            ok = val in values
        else:
            ok = False
        if not ok:
            return False
    return True


def bam_decode(rec, ref_len, split=False, params=None, seqnames=None):
    """Alignment records (inflated, header stripped) -> chrom, start, end, strand in file order,
    or -- params with `which` -- in the order of the which ranges.  params: None (readGAlignments'
    default) or a dict of the ScanBamParam filters (module docstring, items 1-6); `seqnames` (the
    header's reference names) is needed for `which`."""
    params = params or {}
    keep0, keep1 = params.get("flag") or (0xfff, 0xfff)
    keep1 &= ~0x4                                       # bamFlagAND(isUnmappedQuery = FALSE)
    mapq_min = params.get("mapqFilter")
    simple = params.get("simpleCigar", False)
    tag_filter = params.get("tagFilter") or {}
    which = params.get("which")
    kept = []                                           # (ref, pos0, rlen, strand, ranges) in file order
    keys = []
    p = 0
    while p < len(rec):
        bs, ref, pos, l_name, mapq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiiBBHHHi", rec, p)
        q = p + 36 + l_name
        ops = struct.unpack_from("<%dI" % n_cig, rec, q)
        aux = rec[q + 4 * n_cig + (l_seq + 1) // 2 + l_seq:p + 4 + bs]
        p += 4 + bs
        keys.append((1 << 64) - 1 if ref < 0 else (ref << 32) | (pos + 1))
        if (flag & 4) or ref < 0 or pos < 0:
            continue
        if n_cig == 0:
            raise ValueError("a mapped record has no CIGAR")
        if any((c & 15) > 8 for c in ops):
            raise ValueError("CIGAR operation code above 8")
        ok = all(((flag >> b) & 1 and (keep1 >> b) & 1) or (not (flag >> b) & 1 and (keep0 >> b) & 1)
                 for b in range(12))
        ok = ok and (mapq_min is None or mapq >= mapq_min)
        ok = ok and (not simple or (n_cig == 1 and ops[0] & 15 == 0))
        if tag_filter:
            ok = _tags_pass(parse_aux(bytes(aux)), tag_filter) and ok
        if not ok:
            continue
        rlen = sum(c >> 4 for c in ops if (c & 15) in REF_OPS)
        kept.append((ref, pos, max(rlen, 1), -1 if flag & 16 else 1, _ranges_of(ref, pos, ops, int(ref_len[ref]), split)))
    out = []
    if which is None:
        for ref, _, _, st, rr in kept:
            out += [(ref, s, e, st) for s, e in rr]
    else:
        if any(b < a for a, b in zip(keys, keys[1:])):
            raise ValueError("which needs records sorted by (refID, POS)")
        levels = params.get("which_levels") or list(dict.fromkeys(c for c, _, _ in which))
        lut = {c: i for i, c in enumerate(seqnames)}
        for c, s, e in sorted(which, key=lambda x: levels.index(x[0])):
            if c not in lut:
                raise ValueError("which: seqname %s is not in the header" % c)
            if s < 1 or e < s or e > 536870912:
                raise ValueError("which: bad range")
            for ref, pos, rlen, st, rr in kept:
                if ref == lut[c] and pos < e and pos + rlen > s - 1:
                    out += [(ref, a, b, st) for a, b in rr]
    cols = list(zip(*out)) if out else [[], [], [], []]
    return (np.asarray(cols[0], dtype=np.int32), np.asarray(cols[1], dtype=np.int32),
            np.asarray(cols[2], dtype=np.int32), np.asarray(cols[3], dtype=np.int8))
