"""Test helper next to tests/bam_writer.py: alignment records with a chosen MAPQ and typed aux
fields (SAMv1 section 4.2.4).  Like bam_writer, it only ever WRITES the format."""
import struct

from tests.bam_writer import bam_record as _bam_record

AUX_FMT = {"A": "c", "c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}


def bam_record(ref, pos0, flag, cigar, name=b"r", l_seq=0, tags=b"", mapq=30):
    """bam_writer.bam_record with the MAPQ byte (offset 13: after block_size, refID, pos and
    l_read_name) set to `mapq`."""
    rec = _bam_record(ref, pos0, flag, cigar, name=name, l_seq=l_seq, tags=tags)
    return rec[:13] + bytes([mapq]) + rec[14:]


def aux_field(tag, ty, value, sub=None):
    """One typed aux field: ty in A c C s S i I f Z H B; for B, `sub` is the element type
    (c C s S i I f) and `value` the list of elements."""
    head = tag.encode("ascii") + ty.encode("ascii")
    if ty == "A":
        return head + value.encode("ascii")
    if ty in AUX_FMT:
        return head + struct.pack("<" + AUX_FMT[ty], value)
    if ty in "ZH":
        return head + value.encode("ascii") + b"\x00"
    if ty == "B":
        return head + sub.encode("ascii") + struct.pack("<I", len(value)) + struct.pack("<%d%s" % (len(value), AUX_FMT[sub]), *value)
    raise ValueError("aux type %r" % ty)
