"""BigWig input on the device: load, signal coverage and the profile matrix over FLOAT32 coverage.

Two seeded tracks over hg19 are written in memory (tests/bigwig_writer.py, zlib blocks of 1024
items, the bedGraphToBigWig / wigToBigWig default):
    dense   fixedStep, step = span = 25, every base of every chromosome (~1.2e8 items)
    peaks   bedGraph peaks of 200-2000 bp (~2e6 items)
Rows (each after a warm-up; the card's name and power limit are read in the same run):
    load          rcp_bigwig_load wall clock (host parse + inflate on all cores, upload, expand +
                  validation, one host synchronisation), and the same with one inflate thread
    coverage      rcp_signal_coverage over C2's windows (workloads.chipseq_tss: 20 k x 10 kb),
                  CUDA events on the library stream; bytes = 4 * sum(L) written + the items read
    profile       rcp_profile_matrix at 200 bins on that FLOAT32 coverage into a device matrix, next
                  to the same call on an INT32 coverage of the same windows (C2's reads); bytes =
                  4 * sum(L) read + the 8-byte cells written
Shares of peak use the 6 456 GB/s HBM figure the project's other tables use.  100 seeded
windows are checked against oracle/bigwig_oracle.py.

    python tools/bench_bigwig.py [--reps R] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import struct
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_GBS = 6456.0
SLOT = 1024


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:
        return {"name": "unknown (%s)" % e, "power_limit": "unknown"}


def dense_track(chroms, seed=21, span=25):
    """fixedStep sections of SLOT values; values quantised to 0.01 like fold-change tracks."""
    rng = np.random.default_rng(seed)
    secs, items = [], []
    for c, (_, size) in enumerate(chroms):
        n = size // span
        vals = np.round(rng.gamma(1.5, 2.0, size=n), 2).astype(np.float32)
        for k0 in range(0, n, SLOT):
            v = vals[k0:k0 + SLOT]
            start = k0 * span
            end = start + (len(v) - 1) * span + span
            raw = struct.pack("<IIIIIBBH", c, start, end, span, span, 3, 0, len(v)) + v.tobytes()
            secs.append(dict(raw=raw, box=(c, start, c, end)))
        items.append((c, np.arange(n, dtype=np.int64) * span + 1, np.arange(1, n + 1, dtype=np.int64) * span, vals))
    return secs, items


def peak_track(chroms, seed=22, n_peaks=2_000_000):
    rng = np.random.default_rng(seed)
    total = sum(s for _, s in chroms)
    secs, items = [], []
    for c, (_, size) in enumerate(chroms):
        k = int(n_peaks * size / total)
        gap = size // max(k, 1)
        w = rng.integers(200, min(2000, gap - 1), size=k)
        s0 = np.arange(k, dtype=np.int64) * gap + rng.integers(0, gap - w)
        e0 = s0 + w
        v = np.round(rng.gamma(2.0, 5.0, size=k), 3).astype(np.float32)
        rows = np.zeros(k, dtype=[("s", "<u4"), ("e", "<u4"), ("v", "<f4")])
        rows["s"], rows["e"], rows["v"] = s0, e0, v
        for k0 in range(0, k, SLOT):
            r = rows[k0:k0 + SLOT]
            raw = struct.pack("<IIIIIBBH", c, int(r["s"][0]), int(r["e"][-1]), 0, 0, 1, 0, len(r)) + r.tobytes()
            secs.append(dict(raw=raw, box=(c, int(r["s"][0]), c, int(r["e"][-1]))))
        items.append((c, s0 + 1, e0, v))
    return secs, items


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON here (profiles/bigwig_b200.json)")
    args = ap.parse_args()
    import torch
    import recoup_b200 as rb
    import workloads
    from oracle import bigwig_oracle as BO
    from recoup_b200 import _lib
    from tests.bigwig_writer import write_bigwig
    L = _lib.lib
    rb.init(0)
    res = {"card": card(), "peak_gbs": PEAK_GBS, "host_threads": os.cpu_count(), "rows": {}}
    chroms = workloads.HG19
    sizes = [s for _, s in chroms]
    w = workloads.chipseq_tss()
    flank = w["flank"][0]
    ws = (w["region_start"].astype(np.int64) - flank)
    we = (w["region_end"].astype(np.int64) + flank)
    strand = np.ascontiguousarray(w["region_strand"], dtype=np.int8)
    chrom = np.ascontiguousarray(w["region_chrom"], dtype=np.int32)
    ws32, we32 = ws.astype(np.int32), we.astype(np.int32)
    stream = C.c_void_p(L.rcp_stream())
    ext = torch.cuda.ExternalStream(stream.value)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()                                  # warm-up
        L.rcp_sync()
        times = []
        for _ in range(args.reps):
            ev0.record(ext)
            fn()
            ev1.record(ext)
            ev1.synchronize()
            times.append(ev0.elapsed_time(ev1))
        return float(np.median(times)), float(np.min(times))

    for name, maker in (("dense_fixedstep25", dense_track), ("peaks_bedgraph", peak_track)):
        t0 = time.perf_counter()
        secs, items = maker(chroms)
        data = write_bigwig(chroms, secs)
        n_items = sum(len(x[1]) for x in items)
        row = {"items": n_items, "file_bytes": len(data), "write_s": time.perf_counter() - t0}
        buf = np.frombuffer(data, dtype=np.uint8)
        h = C.c_int(0)
        for threads, key in ((0, "load_all_threads"), (1, "load_1_thread")):
            walls = []
            for rep in range(3 if threads == 0 else 1):
                t0 = time.perf_counter()
                _lib.check(L.rcp_bigwig_load(buf.ctypes.data_as(C.c_void_p), buf.shape[0], threads, C.byref(h)))
                walls.append(time.perf_counter() - t0)
                L.rcp_signal_free(h.value)
            row[key] = {"threads": threads or os.cpu_count(), "wall_s_min": min(walls), "wall_s": walls}
        _lib.check(L.rcp_bigwig_load(buf.ctypes.data_as(C.c_void_p), buf.shape[0], 0, C.byref(h)))
        sig = h.value
        cov = C.c_int(0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)

        def coverage():
            _lib.check(L.rcp_signal_coverage(sig, len(chrom), None, p(chrom), p(ws32), p(we32), p(strand),
                                             _lib.MEM_HOST, C.byref(cov)))
            L.rcp_coverage_free(cov.value)
        med, best = timed(coverage)
        _lib.check(L.rcp_signal_coverage(sig, len(chrom), None, p(chrom), p(ws32), p(we32), p(strand),
                                         _lib.MEM_HOST, C.byref(cov)))
        covl = rb.CoverageList(cov.value)
        sum_l = covl.total_len
        oracle = BO.Track(np.concatenate([np.full(len(x[1]), x[0]) for x in items]),
                          np.concatenate([x[1] for x in items]), np.concatenate([x[2] for x in items]),
                          np.concatenate([x[3] for x in items]), sizes)
        # bytes: the output words + the 12-byte items that overlap the non-NULL windows, read once
        live = np.asarray(covl.lengths()) > 0
        under = 0
        for c in range(len(sizes)):
            on = live & (chrom == c)
            a, b = oracle.ptr[c], oracle.ptr[c + 1]
            under += int((np.searchsorted(oracle.start[a:b], we[on], "right") -
                          np.searchsorted(oracle.end[a:b], ws[on], "left")).sum())
        byts = 4 * sum_l + 12 * under
        row["coverage"] = {"ms_median": med, "ms_min": best, "sum_L": sum_l, "items_under_windows": under,
                           "bytes": byts, "share_of_peak": byts / (med * 1e-3) / (PEAK_GBS * 1e9)}
        # oracle check on 100 seeded windows
        rng = np.random.default_rng(5)
        pick = rng.choice(len(chrom), size=100, replace=False)
        want = BO.calc_coverage(oracle, dict(chrom=chrom[pick], start=ws[pick], end=we[pick], strand=strand[pick]))
        got = [covl[int(i)] for i in pick]
        ok = all((a is None and b is None) or (a is not None and b is not None and
                                               np.array_equal(a.view(np.uint32), b.view(np.uint32)))
                 for a, b in zip(got, want))
        row["oracle_100_windows_bit_exact"] = bool(ok)
        # profile matrix, 200 bins, on this FLOAT32 coverage
        R = len(chrom)
        out = torch.empty(200 * R, dtype=torch.float64, device="cuda")

        def profile(hc):
            return lambda: _lib.check(L.rcp_profile_matrix(hc, 1, flank, flank, 0, 200, 0, 0, 42, 0,
                                                           C.c_void_p(out.data_ptr()), R, _lib.MEM_DEVICE))
        med, best = timed(profile(cov.value))
        pb = 4 * sum_l + 8 * R * 200
        row["profile_f32"] = {"ms_median": med, "ms_min": best, "bytes": pb,
                              "share_of_peak": pb / (med * 1e-3) / (PEAK_GBS * 1e9)}
        covl.free()
        L.rcp_signal_free(sig)
        res["rows"][name] = row
        print(json.dumps({name: row}), flush=True)
    # the same profile call on an INT32 coverage of the same windows (C2's reads)
    reads = rb.GRanges(w["read_chrom"], w["read_start"], w["read_end"], strand=w["read_strand"],
                       seqlevels=w["chrom_names"], seqlengths=w["chrom_len"])
    mask = rb.GRanges(chrom, ws32, we32, strand=strand, seqlevels=w["chrom_names"])
    icov = rb.calcCoverage(reads, mask, frag_len=w["frag_len"])
    R = len(chrom)
    out = torch.empty(200 * R, dtype=torch.float64, device="cuda")
    med, best = timed(lambda: _lib.check(L.rcp_profile_matrix(icov.handle, 1, flank, flank, 0, 200, 0, 0, 42, 0,
                                                              C.c_void_p(out.data_ptr()), R, _lib.MEM_DEVICE)))
    pb = 4 * icov.total_len + 8 * R * 200
    res["rows"]["profile_int32_c2"] = {"ms_median": med, "ms_min": best, "sum_L": icov.total_len, "bytes": pb,
                                       "share_of_peak": pb / (med * 1e-3) / (PEAK_GBS * 1e9)}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
