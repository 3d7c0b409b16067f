"""Narrow (uint16) against int32 coverage storage of the split path, in ONE process on the same
inputs: the RCP_COVERAGE_WIDE knob is flipped between alternating rounds of coverageRef +
profileMatrix, and the library's stage timers give sp_tile and prof_bin per round.  Prints one JSON
line: per-stage milliseconds (median over rounds) and the bandwidth those two stages reach at the
bytes each layout stores per covered base (2 or 4).

    python tools/bench_coverage_storage.py --workload C2 --rounds 5 --steps 5
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import workloads as W  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="C2", choices=["C2", "C3"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=5, help="rounds per layout, alternating")
    ap.add_argument("--steps", type=int, default=5, help="coverage + matrix passes per round")
    args = ap.parse_args()

    import torch
    import recoup_b200 as rb
    from recoup_b200 import _lib
    from recoup_b200.coverage import getRegionalRanges

    if not torch.cuda.is_available():
        sys.exit("no GPU: this tool measures on the device")
    rb.init(0)
    L = _lib.lib
    w = W.CONFIGS[args.workload](scale=args.scale)
    lv = list(w["chrom_names"])
    reads = rb.GRanges(w["read_chrom"], w["read_start"], w["read_end"], strand=w["read_strand"],
                       seqlevels=lv, seqlengths=w["chrom_len"])
    genes = rb.GRanges(w["region_chrom"].astype(np.int32), w["region_start"], w["region_end"],
                       strand=w["region_strand"], seqlevels=lv)
    windows = getRegionalRanges(genes, w["region"], w["flank"])
    frag = int(w.get("frag_len", 0))

    def step():
        cov = rb.calcCoverage(reads, windows, frag_len=frag)
        inp = [dict(id="s", name="s", coverage=cov)]
        rb.profileMatrix(inp, w["flank"], w["bin_params"])
        return cov

    n_st = 0
    while L.rcp_timing_stage_name(n_st):
        n_st += 1

    def stages():
        ms = (C.c_double * n_st)()
        cnt = (C.c_int64 * n_st)()
        _lib.check(L.rcp_timing_read(1, n_st, ms, cnt))
        return {L.rcp_timing_stage_name(i).decode(): ms[i] / args.steps for i in range(n_st) if cnt[i] > 0}

    runs = {"narrow": [], "wide": []}
    info = {}
    for mode in ("narrow", "wide"):            # warm-up of both layouts
        os.environ.pop("RCP_COVERAGE_WIDE", None)
        if mode == "wide":
            os.environ["RCP_COVERAGE_WIDE"] = "1"
        cov = step()
        b = C.c_int(0)
        _lib.check(L.rcp_coverage_storage_bytes(cov.handle, C.byref(b)))
        info[mode] = {"bytes_per_base": b.value, "covered_bases": int(cov.lengths().sum())}
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for mode in ("narrow", "wide"):
            os.environ.pop("RCP_COVERAGE_WIDE", None)
            if mode == "wide":
                os.environ["RCP_COVERAGE_WIDE"] = "1"
            _lib.check(L.rcp_timing_enable(1))
            _lib.check(L.rcp_timing_read(1, 0, None, None))
            for _ in range(args.steps):
                step()
            torch.cuda.synchronize()
            runs[mode].append(stages())
            _lib.check(L.rcp_timing_enable(0))
    os.environ.pop("RCP_COVERAGE_WIDE", None)
    out = {"workload": args.workload, "gpu": torch.cuda.get_device_name(0), "rounds": args.rounds,
           "steps": args.steps}
    for mode, rs in runs.items():
        names = sorted(set().union(*rs))
        med = {k: float(np.median([r.get(k, 0.0) for r in rs])) for k in names}
        spread = {k: float(np.ptp([r.get(k, 0.0) for r in rs])) for k in ("sp_tile", "prof_bin") if k in med}
        bw = {k: info[mode]["covered_bases"] * info[mode]["bytes_per_base"] / (med[k] * 1e-3) / 1e9
              for k in ("sp_tile", "prof_bin") if med.get(k)}
        out[mode] = dict(info[mode], stage_ms=med, stage_spread_ms=spread, stored_GBps=bw,
                         total_ms=sum(med.values()))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
