"""Decode rate of the BAM reader under ScanBamParam filters (rcp_bam_decode_param) next to the plain
decode (rcp_bam_decode), on ~2e6 synthetic position-sorted records already in HBM.

Records are shaped like bench.py's import config (36-byte core, 12-byte name, 40M 1000N 35M,
38 bytes of sequence / qualities) plus the aux fields an aligner writes: NM:i, NH:i (1..3), MD:Z
and one B:i array of three elements.  Each row is timed with CUDA events on the library stream
after warm-up, the host synchronisation and the allocations of the call included.

    python tools/bench_bam_params.py [--records N] [--reps R] [--out FILE]

Prints one JSON object (and writes it to --out): per row ms, records/s, record-bytes/s, ranges
out, with the card's name and power limit read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CLEN = np.asarray([249250621, 243199373, 198022430], dtype=np.int64)
NAMES = ["chr1", "chr2", "chr3"]


def make_records(n, seed=9):
    rng = np.random.default_rng(seed)
    name_len, n_cig, l_seq = 21, 3, 19             # 12-byte name and 38-byte tail of bench.py, regrouped
    md = b"MDZ40A34\x00"
    aux_len = 7 + 7 + len(md) + 8 + 12             # NM:i, NH:i, MD:Z, XB:B:i with three elements
    body = 32 + name_len + 4 * n_cig + (l_seq + 1) // 2 + l_seq + aux_len
    rec = np.zeros((n, 4 + body), dtype=np.uint8)

    def v32(col, arr):
        rec[:, col:col + 4] = np.ascontiguousarray(arr, dtype="<i4").view(np.uint8).reshape(n, 4)

    ref = rng.integers(0, 3, size=n)
    pos = (rng.random(n) * (CLEN[ref] - 2000)).astype(np.int64)
    order = np.lexsort((pos, ref))                 # position-sorted
    ref, pos = ref[order], pos[order]
    v32(0, np.full(n, body))
    v32(4, ref)
    v32(8, pos)
    rec[:, 12] = name_len
    rec[:, 13] = rng.integers(0, 61, size=n)       # MAPQ
    rec[:, 16] = n_cig
    flag = rng.choice(np.asarray([0, 16, 1024, 1040, 256, 4], dtype=np.int64), size=n,
                      p=[0.42, 0.42, 0.05, 0.05, 0.04, 0.02])
    rec[:, 18] = flag & 0xff
    rec[:, 19] = flag >> 8
    v32(20, np.full(n, l_seq))
    cig0 = 36 + name_len
    for k, (ln, op) in enumerate(((40, 0), (1000, 3), (35, 0))):
        v32(cig0 + 4 * k, np.full(n, (ln << 4) | op))
    a = cig0 + 4 * n_cig + (l_seq + 1) // 2 + l_seq
    rec[:, a:a + 3] = np.frombuffer(b"NMi", dtype=np.uint8)
    v32(a + 3, rng.integers(0, 4, size=n))
    rec[:, a + 7:a + 10] = np.frombuffer(b"NHi", dtype=np.uint8)
    v32(a + 10, rng.integers(1, 4, size=n))
    rec[:, a + 14:a + 14 + len(md)] = np.frombuffer(md, dtype=np.uint8)
    b = a + 14 + len(md)
    rec[:, b:b + 4] = np.frombuffer(b"XBBi", dtype=np.uint8)
    v32(b + 4, np.full(n, 3))
    for k in range(3):
        v32(b + 8 + 4 * k, rng.integers(-5, 5, size=n))
    assert b + 20 == 4 + body
    return rec.reshape(-1), np.arange(n + 1, dtype=np.int64) * (4 + body)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:          # the rates are still measured; the card is then unknown
        return {"name": "unknown (%s)" % e, "power_limit": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    import recoup_b200 as rb
    from recoup_b200 import _lib
    from recoup_b200.readers import ScanBamParam, bam_decode_param, scanBamFlag
    rb.init(0)
    L = _lib.lib
    rec, off = make_records(args.records)
    n = off.shape[0] - 1
    d_rec = torch.from_numpy(rec).cuda()
    d_off = torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(L.rcp_stream())
    vp = lambda t: C.c_void_p(t.data_ptr())
    clen_p = CLEN.ctypes.data_as(C.POINTER(C.c_int64))
    rng = np.random.default_rng(4)
    starts = [(NAMES[c], int(s)) for c, s in zip(np.sort(rng.integers(0, 3, size=10000)),
                                                   rng.random(10000) * 1.9e8 + 1)]
    rows = {
        "rcp_bam_decode": None,
        "param_all_na": ScanBamParam(),
        "flag_mapq": ScanBamParam(flag=scanBamFlag(isDuplicate=False, isSecondaryAlignment=False), mapqFilter=10),
        "tagFilter_NH_1": ScanBamParam(tagFilter={"NH": [1]}),
        "which_1e4_ranges_10kb": ScanBamParam(which=[(c, s, s + 9999) for c, s in starts]),
        "which_whole_chr1": ScanBamParam(which=[("chr1", 1, int(CLEN[0]))]),
    }

    def decode(params, split):
        h, no = C.c_int(0), C.c_int64(0)
        if params is None:
            _lib.check(L.rcp_bam_decode(vp(d_rec), rec.shape[0], vp(d_off), n, 3, clen_p, split, _lib.MEM_DEVICE,
                                        C.byref(h), C.byref(no)))
        else:
            _lib.check(bam_decode_param(vp(d_rec), rec.shape[0], vp(d_off), n, NAMES, CLEN, split, _lib.MEM_DEVICE,
                                        params, h, no))
        L.rcp_decoded_free(h.value)
        return no.value

    out = {"card": card(), "records": n, "record_bytes": int(rec.shape[0]), "reps": args.reps, "rows": {}}
    for split in (0, 1):
        for key, params in rows.items():
            for _ in range(3):
                decode(params, split)
            L.rcp_sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.reps):
                ranges = decode(params, split)
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / args.reps
            out["rows"]["%s/%s" % (key, "split" if split else "keep")] = {
                "ms": ms, "records_per_s": n / (ms * 1e-3), "record_GB_per_s": rec.shape[0] / (ms * 1e6),
                "ranges_out": ranges}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
