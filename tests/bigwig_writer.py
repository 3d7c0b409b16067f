"""A small, independent bigWig writer (UCSC bbi format, little-endian), built from the layouts of
Kent et al. 2010 and UCSC's bbiFile.h / bwgInternal.h with `struct` and `zlib` only.  It exists to
make test inputs for the library's reader; its own bytes are pinned by the hand-assembled file in
tests/test_bigwig.py.

A section is one data block.  Sections are dicts with `chrom` (id), `type` and:
    "bedGraph"   items = [(start0, end0, value), ...]
    "varStep"    items = [(start0, value), ...], span
    "fixedStep"  items = [value, ...], start (0-based), step, span
Coordinates are 0-based half-open, as in the file.  Sections must be given in (chrom, start)
order.  Options: zlib-compressed or stored blocks, the block sizes of the chromosome B+ tree and
of the R-tree (small sizes give trees of several levels), and zoom headers (written, not used).
"""
import struct
import zlib

BIGWIG_MAGIC = 0x888FFC26
CHROM_TREE_MAGIC = 0x78CA8C91
RTREE_MAGIC = 0x2468ACE0
TYPES = {"bedGraph": 1, "varStep": 2, "fixedStep": 3}


def section_bytes(sec):
    """The 24-byte section header followed by the items (a section may also come as `raw`
    bytes with its `box`, (chrom, start, chrom, end), already packed)."""
    if "raw" in sec:
        return sec["raw"], sec["box"]
    t = TYPES[sec["type"]]
    items = sec["items"]
    step = span = 0
    if t == 1:
        body = b"".join(struct.pack("<IIf", s, e, v) for s, e, v in items)
        start, end = items[0][0], items[-1][1]
    elif t == 2:
        span = sec["span"]
        body = b"".join(struct.pack("<If", s, v) for s, v in items)
        start, end = items[0][0], items[-1][0] + span
    else:
        step, span = sec["step"], sec["span"]
        body = b"".join(struct.pack("<f", v) for v in items)
        start = sec["start"]
        end = start + (len(items) - 1) * step + span
    head = struct.pack("<IIIIIBBH", sec["chrom"], start, end, step, span, t, 0, len(items))
    return head + body, (sec["chrom"], start, sec["chrom"], end)


def _levels(n_items, block):
    """Node counts per level, leaves first, up to one root."""
    levels = [max(1, -(-n_items // block))]
    while levels[-1] > 1:
        levels.append(-(-levels[-1] // block))
    return levels


def _tree(leaf_items, block, leaf_size, inner_size, inner_item, base):
    """Nodes written root first, every node padded to `block` slots.  leaf_items: packed leaf
    entries; inner_item(first, last, child_offset) packs a non-leaf entry for the child whose
    leaf entries run from index first to last.  Returns the bytes; the root is at `base`."""
    levels = _levels(len(leaf_items), block)
    top = len(levels) - 1
    sizes = [4 + block * (leaf_size if lv == 0 else inner_size) for lv in range(len(levels))]
    offsets, pos = {}, base
    for lv in range(top, -1, -1):
        offsets[lv] = pos
        pos += levels[lv] * sizes[lv]
    span = [block ** (lv + 1) for lv in range(len(levels))]       # leaf entries under one node
    out = []
    for lv in range(top, -1, -1):
        for node in range(levels[lv]):
            first = node * span[lv]
            if lv == 0:
                ents = leaf_items[first:first + block]
                body = b"".join(ents)
                size = leaf_size
            else:
                ents = []
                for k in range(block):
                    child = node * block + k
                    if child >= levels[lv - 1]:
                        break
                    a = child * span[lv - 1]
                    b = min(a + span[lv - 1], len(leaf_items)) - 1
                    ents.append(inner_item(a, b, offsets[lv - 1] + child * sizes[lv - 1]))
                body = b"".join(ents)
                size = inner_size
            out.append(struct.pack("<BBH", 1 if lv == 0 else 0, 0, len(ents)) + body)
            out.append(b"\0" * ((block - len(ents)) * size))
    return b"".join(out)


def write_bigwig(chroms, sections, compress=True, chrom_block=256, rtree_block=256, zoom_levels=0,
                 items_per_slot=1024):
    """chroms: [(name, size)] in chromId order.  Returns the file's bytes."""
    zoom = b"".join(struct.pack("<IIQQ", 4 ** (i + 2), 0, 0xDEADBEEF, 0xFEEDFACE) for i in range(zoom_levels))
    chrom_tree_off = 64 + len(zoom)
    key_size = max(len(n.encode()) for n, _ in chroms)
    order = sorted(range(len(chroms)), key=lambda i: chroms[i][0].encode())
    keys = [chroms[i][0].encode().ljust(key_size, b"\0") for i in order]
    leaves = [keys[k] + struct.pack("<II", order[k], chroms[order[k]][1]) for k in range(len(order))]
    block = min(chrom_block, len(chroms))
    tree = _tree(leaves, block, key_size + 8, key_size + 8,
                 lambda a, b, off: keys[a] + struct.pack("<Q", off), chrom_tree_off + 32)
    chrom_tree = struct.pack("<IIIIQQ", CHROM_TREE_MAGIC, block, key_size, 8, len(chroms), 0) + tree
    data_off = chrom_tree_off + len(chrom_tree)
    data = [struct.pack("<Q", len(sections))]
    blocks, boxes, max_raw, pos = [], [], 0, data_off + 8
    for sec in sections:
        raw, box = section_bytes(sec)
        max_raw = max(max_raw, len(raw))
        payload = zlib.compress(raw) if compress else raw
        blocks.append((pos, len(payload)))
        boxes.append(box)
        data.append(payload)
        pos += len(payload)
    data = b"".join(data)
    index_off = data_off + len(data)
    leaves = [struct.pack("<IIIIQQ", *boxes[i], blocks[i][0], blocks[i][1]) for i in range(len(blocks))]

    def inner(a, b, off):
        return struct.pack("<IIIIQ", boxes[a][0], boxes[a][1], boxes[b][2], boxes[b][3], off)

    rblock = min(rtree_block, max(len(blocks), 1))
    rtree = _tree(leaves, rblock, 32, 24, inner, index_off + 48)
    first, last = (boxes[0], boxes[-1]) if boxes else ((0, 0, 0, 0), (0, 0, 0, 0))
    index = struct.pack("<IIQIIIIQII", RTREE_MAGIC, rblock, len(blocks), first[0], first[1], last[2], last[3],
                        index_off, items_per_slot, 0) + rtree
    header = struct.pack("<IHHQQQHHQQIQ", BIGWIG_MAGIC, 4, zoom_levels, chrom_tree_off, data_off, index_off,
                         0, 0, 0, 0, max_raw if compress else 0, 0)
    assert len(header) == 64
    return header + zoom + chrom_tree + data + index


def items_of(sections):
    """(chrom, start0, end0, value) of every item, in section order."""
    out = []
    for sec in sections:
        t = TYPES[sec["type"]]
        for i, it in enumerate(sec["items"]):
            if t == 1:
                out.append((sec["chrom"], it[0], it[1], it[2]))
            elif t == 2:
                out.append((sec["chrom"], it[0], it[0] + sec["span"], it[1]))
            else:
                s = sec["start"] + i * sec["step"]
                out.append((sec["chrom"], s, s + sec["span"], it))
    return out
