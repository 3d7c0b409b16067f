#!/usr/bin/env python
"""bench.py -- reads -> coverage -> profile matrix on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2|C3|C4|C5] [--scale S]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      (CPU arm: the oracle's C port on the host cores)

A "step" is one pass of the hot path over one sample: rcp_reads_load (global-coordinate map) ->
rcp_coverage (exact per-base int32 coverage of every region) -> rcp_profile_matrix (regions x
bins fp64, column-major) [-> NCCL gather of the row blocks to rank 0 when N > 1].  `value` times
that with the decoded reads/regions already resident in HBM; `e2e` times the same through the
public host API with pinned HOST buffers, copies included.

The JSON line carries, beside the headline (C2):
  configs   C1, C3 (all 8 samples), C4, C5 of BASELINE.json at full size, one GPU (N = 1 only)
  fused     the C2 step through rcp_coverage_profile (coverage not materialised)
  strong    ONE C5 problem sharded by region over the N ranks: reads exchanged with an NCCL
            all-to-all inside the timed region, each rank's matrix block downloaded over its own
            PCIe link; `checksum` is the same for every N
For N > 1 the headline itself is N independent C2 replicas (weak scaling: every rank a full-size
sample of its own) whose row blocks are gathered to rank 0.
"""
import argparse
import ctypes as C
import datetime
import json
import os
import queue
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads as W  # noqa: E402

METRIC = "reads/s through coverage + profileMatrix (reads -> per-base coverage -> regions x bins)"
UNIT = "reads/s"
SEEDS = {"C2": 1001, "C3": 1003, "C4": 1004, "C5": 1005}
PATHS = {0: "list", 1: "index", 2: "buckets", 3: "blocks", 4: "split"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(W.CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="all", choices=["all", "none"],
                    help="N = 1: also run C1, C3, C4 and C5 (device-resident) and report them in `configs`")
    ap.add_argument("--configs-scale", type=float, default=1.0,
                    help="scale of the extra configs and of the strong-scaling problem (1.0 = the named sizes)")
    ap.add_argument("--strong", default="on", choices=["on", "off"],
                    help="also run ONE C5 problem sharded by region over the N ranks (`strong` in the line)")
    ap.add_argument("--read-order", default="random", choices=["random", "coordinate"],
                    help="order of the synthetic reads: as generated (random; the default and the "
                         "harder case) or sorted by chromosome and start like a coordinate-sorted BAM")
    ap.add_argument("--exchange", default="ce", choices=["ce", "nccl"],
                    help="N > 1: how the row blocks reach rank 0 -- ce: every rank puts its block "
                         "straight into rank 0's matrix (CUDA IPC mapping) with the copy engine over "
                         "NVLink + a one-word NCCL all-reduce as the fence; nccl: dist.gather + placement")
    ap.add_argument("--path", default="auto", choices=["auto", "index", "buckets", "blocks", "split"],
                    help="rcp_set_coverage_path: how rcp_coverage finds each region's reads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the profile matrix of the last timed step (rank 0: the "
                         "gathered matrix) as DIR/profile.npy, regions x bins float64; above 64 MB a fixed, "
                         "seeded sample of its rows. The inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm sizes its sample by a timed "
                 "calibration pass, so its inputs differ from run to run")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 50 ms from before the warm-up until
    after the e2e loop; rows are stamped on arrival so the timed window can be cut out."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t_begin, t_end, label="timed region"):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def digest(rows):
            sm, mx, reasons = [], [], set()
            for _t, row in rows:
                f = [x.strip() for x in row.split(",")]
                if len(f) < 6:
                    continue
                try:
                    sm.append(float(f[0]))
                    mx.append(float(f[1]))
                except ValueError:
                    continue
                for nme, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            return sm, mx, reasons

        inside = [r for r in self.rows if t_begin <= r[0] <= t_end]
        window = label
        if len(inside) < 3:
            inside = self.rows          # timed region shorter than the sampling period
            window = "warm-up + timed region (timed region < 3 samples long)"
        sm, mx, reasons = digest(inside)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port)
# ------------------------------------------------------------------------------------------------
def cpu_pass(w, frac):
    """One pass of the oracle's C port over the first `frac` of the reads and regions of
    workload `w`.  Returns (seconds, reads processed, description)."""
    from oracle import c_oracle as CO
    from oracle import recoup_oracle as O
    n = max(int(len(w["read_start"]) * frac), 1)
    t0 = time.perf_counter()
    ix = CO.Index(w["read_chrom"][:n], w["read_start"][:n], w["read_end"][:n], w["read_strand"][:n],
                  w["chrom_len"], frag_len=w["frag_len"])
    if w["region"] == "rna":
        G = max(int((len(w["exon_ptr"]) - 1) * frac), 1)
        ptr = w["exon_ptr"][:G + 1]
        ne = int(ptr[-1])
        f1, f2 = w["flank"]
        gs, ge, gst, gc = (w["region_start"][:G], w["region_end"][:G], w["region_strand"][:G],
                           w["region_chrom"][:G])
        ls, le = O.get_flanking_ranges(gs, ge, gst, f1, "upstream")
        rs, re_ = O.get_flanking_ranges(gs, ge, gst, f2, "downstream")
        center = CO.coverage_list(ix, ptr, w["exon_chrom"][:ne], w["exon_start"][:ne],
                                  w["exon_end"][:ne], w["exon_strand"][:ne])
        left = CO.coverage(ix, gc, ls, le, gst)
        right = CO.coverage(ix, gc, rs, re_, gst)
        # merge + bins on the list form (python); small next to the coverage passes
        merged = CO.concat3(left.to_list(), center.to_list(), right.to_list())
        O.profile_matrix(merged, w["flank"], w["bin_params"])
        n_units = G
    else:
        R = max(int(len(w["region_start"]) * frac), 1)
        s, e = O.get_regional_ranges(w["region_start"][:R], w["region_end"][:R],
                                     w["region_strand"][:R], w["region"], w["flank"])
        dense = CO.coverage(ix, w["region_chrom"][:R], s, e, w["region_strand"][:R])
        lens = dense.len[dense.len > 0]
        equal = bool((lens == lens[0]).all()) if lens.size else True
        CO.profile_matrix(dense, w["flank"], w["bin_params"], equal)
        n_units = R
    dt = time.perf_counter() - t0
    return dt, n, "first %d reads and %d regions of %s" % (n, n_units, w["name"])


def cpu_baseline(w, budget_s=20.0):
    from oracle import c_oracle as CO
    frac = min(1.0, 2_000_000 / max(len(w["read_start"]), 1))
    dt, n, what = cpu_pass(w, frac)                       # calibration pass
    rate = n / dt
    frac2 = min(1.0, budget_s * rate / len(w["read_start"]))
    if frac2 > frac * 1.5:
        dt, n, what = cpu_pass(w, frac2)
    return {"value": n / dt, "unit": UNIT, "cores": CO.threads(), "kind": "port",
            "sample": what + " (oracle C port, OpenMP over regions; R itself is not installable "
                             "here)", "seconds": round(dt, 3)}


def run_reference(args):
    """--impl reference: the reference's CPU path.  R/Bioconductor cannot run in this image (no
    R, no network), so this arm times the oracle's C/OpenMP port with every host thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if "TORCHELASTIC_RUN_ID" in os.environ or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # torchrun sets OMP_NUM_THREADS=1 for its workers; the CPU arm is meant to use every host
        # thread it can (rank 0 alone works here), so undo that before the OpenMP runtime starts
        os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    w = W.CONFIGS[args.workload](scale=args.scale)
    from oracle import c_oracle as CO
    total = max(len(w["read_start"]), 1)
    frac = min(1.0, 2_000_000 / total)
    dt, n, what = cpu_pass(w, frac)                       # calibration
    per_step_s = min(20.0, 150.0 / max(args.steps + args.warmup, 1))
    frac = min(1.0, max(frac, per_step_s * (n / dt) / total))
    for _ in range(args.warmup):
        cpu_pass(w, frac)
    t = 0.0
    reads = 0
    for _ in range(args.steps):
        dt, n, what = cpu_pass(w, frac)
        t += dt
        reads += n
    val = reads / t
    cb = {"value": val, "unit": UNIT, "cores": CO.threads(), "kind": "port", "sample": what}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/f64",
        "data": "synthetic", "config": {"workload": w["name"], "sample": what},
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Problem:
    """One workload with its reads and regions resident on the device, and the step over it:
    rcp_reads_load -> rcp_coverage[_list / x3 + concat] -> rcp_profile_matrix, all device memory."""

    def __init__(self, env, w, reads=None, region_idx=None):
        import torch
        self.env, self.w = env, w
        rb, dev = env["rb"], env["dev"]
        from recoup_b200.ranges import getFlankingRanges, getRegionalRanges
        self.is_rna = w["region"] == "rna"
        sel = slice(None) if region_idx is None else region_idx
        self.genes = rb.GRanges(w["region_chrom"][sel], w["region_start"][sel], w["region_end"][sel],
                                strand=w["region_strand"][sel], seqlevels=w["chrom_names"])
        self.f1, self.f2 = w["flank"]
        self.bp = w["bin_params"]
        self.clen = np.ascontiguousarray(w["chrom_len"], dtype=np.int64)

        def to_dev(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

        if self.is_rna:
            left = getFlankingRanges(self.genes, self.f1, "upstream")
            right = getFlankingRanges(self.genes, self.f2, "downstream")
            self.R = len(self.genes)
            self.d_left = [to_dev(x) for x in (left.seqnames, left.start, left.end, left.strand)]
            self.d_right = [to_dev(x) for x in (right.seqnames, right.start, right.end, right.strand)]
            self.ex = [np.ascontiguousarray(w[k]) for k in ("exon_chrom", "exon_start", "exon_end", "exon_strand")]
            self.ex_ptr = np.ascontiguousarray(w["exon_ptr"], dtype=np.int64)
        else:
            self.win = getRegionalRanges(self.genes, w["region"], w["flank"])
            self.R = len(self.win)
            self.d_win = [to_dev(x) for x in (self.win.seqnames, self.win.start, self.win.end, self.win.strand)]
        self.equal_lengths = 1 if w["region"] in ("tss", "tes", "custom") else 0
        self.set_reads(reads if reads is not None else
                       [to_dev(w[k]) for k in ("read_chrom", "read_start", "read_end", "read_strand")])
        self.ncols = None
        self.stats = {}
        self.out = None

    def set_reads(self, d_reads):
        self.d_reads = d_reads
        self.N = int(d_reads[1].shape[0])

    def _load(self):
        L, _lib = self.env["L"], self.env["_lib"]
        vp = lambda t: C.c_void_p(t.data_ptr())                # noqa: E731
        h = C.c_int(0)
        r = self.d_reads
        _lib.check(L.rcp_reads_load(self.N, vp(r[0]), vp(r[1]), vp(r[2]), vp(r[3]) if r[3] is not None else None,
                                    self.clen.shape[0], self.clen.ctypes.data_as(C.POINTER(C.c_int64)),
                                    int(self.w["frag_len"]), _lib.MEM_DEVICE, C.byref(h)))
        return h

    def step(self, out_ptr=None, ld=None):
        """reads (HBM) -> coverage -> matrix (HBM).  out_ptr / ld: where the matrix goes (default:
        this problem's own buffer)."""
        import torch
        L, _lib = self.env["L"], self.env["_lib"]
        vp = lambda t: C.c_void_p(t.data_ptr())                # noqa: E731
        hp = lambda a: a.ctypes.data_as(C.c_void_p)            # noqa: E731
        R = self.R
        h = self._load()
        cov = C.c_int(0)
        if self.is_rna:
            hc, hl, hr = C.c_int(0), C.c_int(0), C.c_int(0)
            _lib.check(L.rcp_coverage_list(h.value, R, self.ex_ptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                           hp(self.ex[0]), hp(self.ex[1]), hp(self.ex[2]), hp(self.ex[3]), 1,
                                           _lib.STRAND_ANY, _lib.MEM_HOST, C.byref(hc)))
            dl, dr = self.d_left, self.d_right
            _lib.check(L.rcp_coverage(h.value, R, vp(dl[0]), vp(dl[1]), vp(dl[2]), vp(dl[3]), 1,
                                      _lib.STRAND_ANY, _lib.MEM_DEVICE, C.byref(hl)))
            _lib.check(L.rcp_coverage(h.value, R, vp(dr[0]), vp(dr[1]), vp(dr[2]), vp(dr[3]), 1,
                                      _lib.STRAND_ANY, _lib.MEM_DEVICE, C.byref(hr)))
            _lib.check(L.rcp_coverage_concat3(hl.value, hc.value, hr.value, C.byref(cov)))
            for x in (hc, hl, hr):
                L.rcp_coverage_free(x.value)
        else:
            dw = self.d_win
            _lib.check(L.rcp_coverage(h.value, R, vp(dw[0]), vp(dw[1]), vp(dw[2]), vp(dw[3]), 1,
                                      _lib.STRAND_ANY, _lib.MEM_DEVICE, C.byref(cov)))
        if self.ncols is None:
            nc = C.c_int64(0)
            _lib.check(L.rcp_profile_ncols(cov.value, self.equal_lengths, self.f1, self.f2,
                                           self.bp["flankBinSize"], self.bp["regionBinSize"], C.byref(nc)))
            self.ncols = nc.value
        if out_ptr is None:
            if self.out is None:
                self.out = torch.empty((self.ncols, R), dtype=torch.float64, device=self.env["dev"])
            out_ptr, ld = self.out.data_ptr(), R
        _lib.check(L.rcp_profile_matrix(cov.value, self.equal_lengths, self.f1, self.f2,
                                        self.bp["flankBinSize"], self.bp["regionBinSize"],
                                        _lib.STAT[self.bp["sumStat"]], _lib.INTERP[self.bp["interpolation"]],
                                        42, 0, C.c_void_p(out_ptr), ld, _lib.MEM_DEVICE))
        if not self.stats:
            tl, nn = C.c_int64(0), C.c_int64(0)
            L.rcp_coverage_info(cov.value, None, C.byref(tl), C.byref(nn), None)
            pth, cand = C.c_int(0), C.c_int64(0)
            L.rcp_coverage_path_info(cov.value, C.byref(pth), C.byref(cand))
            self.stats = {"total_len": tl.value, "n_null": nn.value, "path": PATHS[pth.value],
                          "candidates": cand.value}
        L.rcp_coverage_free(cov.value)
        L.rcp_reads_free(h.value)

    def fused_step(self):
        """Equal-length windows only: rcp_coverage_profile (coverage not materialised)."""
        L, _lib = self.env["L"], self.env["_lib"]
        vp = lambda t: C.c_void_p(t.data_ptr())                # noqa: E731
        h = self._load()
        dw = self.d_win
        _lib.check(L.rcp_coverage_profile(h.value, self.R, vp(dw[0]), vp(dw[1]), vp(dw[2]), vp(dw[3]), 1,
                                          _lib.STRAND_ANY, self.bp["regionBinSize"], 42, 0, 1.0,
                                          C.c_void_p(self.out.data_ptr()), self.R, None, _lib.MEM_DEVICE))
        L.rcp_reads_free(h.value)


def stage_table(L, _lib):
    n_st = 0
    while L.rcp_timing_stage_name(n_st):
        n_st += 1
    ms = (C.c_double * n_st)()
    cnt = (C.c_int64 * n_st)()
    _lib.check(L.rcp_timing_read(1, n_st, ms, cnt))
    return {L.rcp_timing_stage_name(i).decode(): (ms[i] / max(cnt[i], 1), int(cnt[i]))
            for i in range(n_st) if cnt[i] > 0}


STAGE_GROUPS = {
    "reads_map": ["index_map"],
    "coverage": ["index_sort", "cov_plan", "cov_tile", "cov_small", "cov_list", "cov_concat",
                 "bkt_plan", "bkt_count", "bkt_scatter", "bkt_tile", "bkt_small",
                 "blk_filter", "blk_hist", "blk_scatter", "blk_tile", "blk_small",
                 "sp_plan", "sp_split", "sp_sort", "sp_tile", "sp_small"],
    "profile": ["prof_bin", "prof_interp", "prof_base"],
}


def stage_roofline(stage, steps, N, R, ncols, total_len, peak):
    """SURVEY 8d algorithmic bytes per STAGE / the stage's whole time (sort / bucketing / planning
    included in the TIME, not in the bytes):
      reads_map  13 B/read in (chrom, start, end, strand) + 9 B/read out
      coverage   8 B/read + 4 B/covered base + 16 B/region
      profile    4 B/covered base + 8 B/matrix cell"""
    nbytes = {"reads_map": 22 * N, "coverage": 8 * N + 4 * total_len + 16 * R,
              "profile": 4 * total_len + 8 * R * ncols}
    per_step = {k: v[0] * v[1] / steps for k, v in stage.items()}
    out = {}
    for g, members in STAGE_GROUPS.items():
        ms_g = sum(per_step.get(m, 0.0) for m in members)
        if ms_g > 0:
            ach = nbytes[g] / (ms_g * 1e-3) / 1e9
            out[g] = {"ms_per_step": ms_g, "algorithmic_bytes": nbytes[g], "achieved": ach, "frac": ach / peak}
    return out, per_step


def time_problem(env, prob, steps, warmup, step_fn=None):
    """W untimed + K timed steps of one problem on the library stream; returns (ms/step, stages)."""
    import torch
    L, _lib, stream = env["L"], env["_lib"], env["stream"]
    fn = step_fn or prob.step
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    _lib.check(L.rcp_timing_enable(1))
    _lib.check(L.rcp_timing_read(1, 0, None, None))
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        fn()
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    stage = stage_table(L, _lib)
    _lib.check(L.rcp_timing_enable(0))
    return ms, stage


def config_entry(env, w, steps, peak, samples=1, note=None):
    """One extra config, device-resident: ms per sample step, stage times and roofline fractions."""
    prob = Problem(env, w)
    ms, stage = time_problem(env, prob, steps, 3)
    roof, per_step = stage_roofline(stage, steps, prob.N, prob.R, prob.ncols, prob.stats["total_len"], peak)
    out = {"workload": w["name"], "reads_per_sample": prob.N, "regions": prob.R, "matrix_cols": prob.ncols,
           "covered_bases": prob.stats["total_len"], "null_regions": prob.stats["n_null"],
           "coverage_path_used": prob.stats["path"], "samples": samples, "steps_per_sample": steps,
           "ms_per_sample": ms, "reads_per_s": prob.N / (ms * 1e-3),
           "region_bins_per_s": prob.R * prob.ncols / (ms * 1e-3),
           "stage_ms": per_step, "stages": roof}
    if note:
        out["note"] = note
    return out


def run_c1(env):
    """C1: the reference's bundled ChIP-seq data (both samples), TSS +-2 kb, 100 bins, through the
    HOST API (the fixture is tiny: latency-bound; parity config)."""
    import torch
    rb = env["rb"]
    z = np.load(os.path.join(ROOT, "tests", "golden", "recoup_test_data.npz"))
    n = z["gene_start"].shape[0]
    genes = rb.GRanges(np.zeros(n, dtype=np.int32), z["gene_start"], z["gene_end"], strand=z["gene_strand"],
                       seqlevels=["chr12"], names=list(z["gene_names"]))
    bp = dict(flankBinSize=0, regionBinSize=100, sumStat="mean", interpolation="auto")
    reads = []
    for k in range(2):
        s = z["reads_%d_start" % k].astype(np.int64)
        wd = z["reads_%d_width" % k].astype(np.int64)
        reads.append(rb.GRanges(np.zeros(s.shape[0], dtype=np.int32), s, s + wd - 1, strand=z["reads_%d_strand" % k],
                                seqlevels=["chr12"], seqlengths=z["chrom_len"]))

    def one():
        inp = [dict(id="s%d" % k, name="s%d" % k, ranges=reads[k]) for k in range(2)]
        rb.coverageRef(inp, genes, "tss", (2000, 2000))
        rb.profileMatrix(inp, (2000, 2000), bp)
        for x in inp:
            x["coverage"].free()
        for g in reads:
            for dr in g._device.values():
                dr.free()
            g._device.clear()
        return inp

    for _ in range(3):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 10
    for _ in range(reps):
        inp = one()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / reps
    nreads = sum(len(r) for r in reads)
    return {"workload": "C1 recoup_test_data: 2 samples x 100000 reads over 100 genes, TSS +-2 kb, 100 bins",
            "through": "host API (coverageRef + profileMatrix), host arrays, copies included",
            "ms_per_pass": ms, "reads_per_s": nreads / (ms * 1e-3), "matrix": list(inp[0]["profile"].shape),
            "note": "latency-bound (0.8 MB of reads): parity config, not a roofline config"}


def run_import(env, n_records=2_000_000):
    """Read import (SURVEY 8f N3): rcp_bam_decode / rcp_bed_decode on synthetic files with the record
    and text bytes already in HBM (device-timed) and from pinned-free host memory (wall clock, copies
    included).  Records: 36-byte core + 12-byte name + 3 CIGAR operations (40M 1000N 35M: spliced
    reads, two ranges each under spliceAction split) + 38 bytes of sequence / qualities."""
    import ctypes as C

    import torch
    _lib = env["_lib"]
    L = _lib.lib
    rng = np.random.default_rng(9)
    clen = np.asarray([249250621, 243199373, 198022430], dtype=np.int64)
    n = int(n_records)
    name_len, n_cig, tail = 12, 3, 38
    body = 32 + name_len + 4 * n_cig + tail
    rec = np.zeros((n, 4 + body), dtype=np.uint8)
    v32 = lambda col, arr: rec.__setitem__((slice(None), slice(col, col + 4)),
                                           np.ascontiguousarray(arr, dtype="<i4").view(np.uint8).reshape(n, 4))
    ref = rng.integers(0, 3, size=n)
    v32(0, np.full(n, body))
    v32(4, ref)
    v32(8, (rng.random(n) * (clen[ref] - 2000)).astype(np.int64))
    rec[:, 12] = name_len
    rec[:, 16] = n_cig
    flag = rng.choice(np.asarray([0, 16, 4], dtype=np.int64), size=n, p=[0.49, 0.49, 0.02])
    rec[:, 18] = flag
    cig0 = 36 + name_len
    for k, (ln, op) in enumerate(((40, 0), (1000, 3), (35, 0))):
        v32(cig0 + 4 * k, np.full(n, (ln << 4) | op))
    rec = rec.reshape(-1)
    n_bytes = rec.shape[0]
    off = np.arange(n + 1, dtype=np.int64) * (4 + body)
    dev = torch.device("cuda", torch.cuda.current_device())
    d_rec = torch.from_numpy(rec).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    vp = lambda t: C.c_void_p(t.data_ptr())
    hp = lambda a: a.ctypes.data_as(C.c_void_p)
    clen_p = clen.ctypes.data_as(C.POINTER(C.c_int64))
    out = {"records": n, "record_bytes": n_bytes}

    def timed(fn, reps=5):
        for _ in range(2):
            fn()
        L.rcp_sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        L.rcp_sync()
        return 1e3 * (time.perf_counter() - t0) / reps

    def bam(mem, split):
        h, no = C.c_int(0), C.c_int64(0)
        if mem == _lib.MEM_DEVICE:
            _lib.check(L.rcp_bam_decode(vp(d_rec), n_bytes, vp(d_off), n, 3, clen_p, split, mem, C.byref(h), C.byref(no)))
        else:
            _lib.check(L.rcp_bam_decode(hp(rec), n_bytes, hp(off), n, 3, clen_p, split, mem, C.byref(h), C.byref(no)))
        L.rcp_decoded_free(h.value)
        return no.value

    for split in (0, 1):
        key = "bam_split" if split else "bam_keep"
        ms = timed(lambda: bam(_lib.MEM_DEVICE, split))
        out[key] = {"ranges_out": bam(_lib.MEM_DEVICE, split), "ms_device_resident": ms,
                    "records_per_s": n / (ms * 1e-3), "GB_per_s": n_bytes / (ms * 1e6)}
    ms = timed(lambda: bam(_lib.MEM_HOST, 0), reps=3)
    out["bam_keep"]["ms_from_host"] = ms
    t0 = time.perf_counter()
    cnt = C.c_int64(0)
    _lib.check(L.rcp_bam_index(hp(rec), n_bytes, C.byref(cnt), hp(off), n + 1))
    out["bam_index_host_ms"] = 1e3 * (time.perf_counter() - t0)
    del d_rec, d_off
    # the BGZF inflate before the decode (host: zlib, one thread per core): 64 MB of the records
    import struct
    import zlib

    def bgzf_block(data):
        comp = zlib.compressobj(1, zlib.DEFLATED, -15)
        body = comp.compress(data) + comp.flush()
        head = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(body) + 25)
        return head + body + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data))

    part = rec[:64 << 20].tobytes()
    bgzf = np.frombuffer(b"".join(bgzf_block(part[i:i + 60000]) for i in range(0, len(part), 60000)) + bgzf_block(b""),
                         dtype=np.uint8)
    inflated = np.empty(len(part), dtype=np.uint8)
    t0 = time.perf_counter()
    _lib.check(L.rcp_bgzf_inflate(hp(bgzf), bgzf.shape[0], hp(inflated), inflated.shape[0], 0))
    dt = time.perf_counter() - t0
    out["bgzf_inflate_host"] = {"compressed_bytes": int(bgzf.shape[0]), "inflated_bytes": len(part), "ms": 1e3 * dt,
                                "GB_per_s_inflated": len(part) / dt / 1e9, "threads": len(os.sched_getaffinity(0)),
                                "matches": bool(np.array_equal(inflated, rec[:64 << 20]))}
    del part, bgzf, inflated
    # BED: six columns, ~33 bytes per line
    m = n
    names = ["chr1", "chr2", "chr3"]
    a = (rng.random(m) * 1.9e8).astype(np.int64)
    cols = [np.asarray(names)[rng.integers(0, 3, size=m)], a.astype(str), (a + 36).astype(str),
            np.full(m, "r"), np.full(m, "0"), np.where(rng.random(m) < 0.5, "+", "-")]
    text = "\n".join(map("\t".join, zip(*cols))).encode() + b"\n"
    t_host = np.frombuffer(text, dtype=np.uint8)
    d_text = torch.from_numpy(t_host.copy()).to(dev)
    arr = (C.c_char_p * 3)(*[s.encode() for s in names])

    def bed(mem):
        h, no = C.c_int(0), C.c_int64(0)
        src = vp(d_text) if mem == _lib.MEM_DEVICE else hp(t_host)
        _lib.check(L.rcp_bed_decode(src, t_host.shape[0], 3, arr, mem, C.byref(h), C.byref(no)))
        L.rcp_decoded_free(h.value)
        return no.value

    ms = timed(lambda: bed(_lib.MEM_DEVICE))
    out["bed"] = {"lines": m, "text_bytes": int(t_host.shape[0]), "ranges_out": bed(_lib.MEM_DEVICE),
                  "ms_device_resident": ms, "lines_per_s": m / (ms * 1e-3), "GB_per_s": t_host.shape[0] / (ms * 1e6),
                  "ms_from_host": timed(lambda: bed(_lib.MEM_HOST), reps=3)}
    out["note"] = ("device rates are decode only: the BGZF inflate (bgzf_inflate_host) and the host walk of the "
                   "record chain (bam_index_host_ms) come before it")
    return out


def run_strong(env, args, world, rank, which="C5"):
    """ONE problem sharded by region -- C5 (every rank generates the read parts {p : p % W == rank})
    or C3 (every rank keeps the reads rank, rank + W, ... of the one seeded sample): an arbitrary
    share of the reads per rank; the timed step exchanges the reads (all-to-all by region slice),
    runs the path on the rank's slice and downloads the rank's matrix block over its own PCIe
    link.  checksum = sum of all matrix entries: the same for every W."""
    import torch
    import torch.distributed as dist
    from recoup_b200.ranges import getRegionalRanges
    from recoup_b200.sharding import exchange_reads, partition_regions, slice_spans
    rb, dev, L = env["rb"], env["dev"], env["L"]
    t_gen = time.time()
    if which == "C5":
        n_parts = 8
        mine = [p for p in range(n_parts) if p % world == rank]
        ws = [W.dnase_sites_part(p, n_parts=n_parts, scale=args.configs_scale) for p in mine]
        w = dict(ws[0])
        for key in ("read_chrom", "read_start", "read_end", "read_strand"):
            w[key] = np.concatenate([x[key] for x in ws])
        del ws
    else:
        w = W.gene_bodies(scale=args.configs_scale, seed=SEEDS["C3"])
        for key in ("read_chrom", "read_start", "read_end", "read_strand"):
            w[key] = np.ascontiguousarray(w[key][rank::world])
    t_gen = time.time() - t_gen
    genes = rb.GRanges(w["region_chrom"], w["region_start"], w["region_end"], strand=w["region_strand"],
                       seqlevels=w["chrom_names"])
    win = getRegionalRanges(genes, w["region"], w["flank"])
    parts = partition_regions(win.seqnames, win.start, win.end, world)
    spans = slice_spans(win.seqnames, win.start, win.end, parts, len(w["chrom_len"]))
    my_idx = np.sort(parts[rank])
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    share = [to_dev(w[k]) for k in ("read_chrom", "read_start", "read_end", "read_strand")]
    n_share = int(share[1].shape[0])
    for key in ("read_chrom", "read_start", "read_end", "read_strand"):
        w[key] = w[key][:0]
    prob = Problem(env, w, reads=share, region_idx=my_idx)
    R_mine = prob.R
    if which == "C5":
        ncols = w["flank"][0] + w["flank"][1]      # per-base custom windows: f1 + f2 columns
    else:
        ncols = 2 * w["bin_params"]["flankBinSize"] + w["bin_params"]["regionBinSize"]
    block = torch.empty((ncols, R_mine), dtype=torch.float64, device=dev)
    host = torch.empty((ncols, R_mine), dtype=torch.float64, pin_memory=True)
    lib_stream = torch.cuda.ExternalStream(L.rcp_stream(), device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def step():
        with torch.cuda.stream(lib_stream):
            ev[0].record(lib_stream)
            got = exchange_reads(share[0], share[1], share[2], share[3], spans, filter_single=False)
            ev[1].record(lib_stream)
            prob.set_reads(list(got))
            prob.step(out_ptr=block.data_ptr(), ld=R_mine)
            ev[2].record(lib_stream)
            host.copy_(block, non_blocking=True)
            ev[3].record(lib_stream)
        torch.cuda.synchronize()
        return int(got[1].shape[0])

    for _ in range(2):
        step()
    if world > 1:
        dist.barrier()
    steps = max(2, min(args.steps, 3))
    phases = np.zeros(3)
    total_ms = 0.0
    n_mine = 0
    _lib = env["_lib"]
    _lib.check(L.rcp_timing_enable(1))
    _lib.check(L.rcp_timing_read(1, 0, None, None))
    for _ in range(steps):
        n_mine = step()
        total_ms += ev[0].elapsed_time(ev[3])
        phases += [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])]
        if world > 1:
            dist.barrier()
    ms = total_ms / steps
    stage = stage_table(L, _lib)
    _lib.check(L.rcp_timing_enable(0))
    checksum = float(host.sum())
    red = torch.tensor([ms, phases[0] / steps, phases[1] / steps, phases[2] / steps], dtype=torch.float64, device=dev)
    tot = torch.tensor([checksum, float(n_share), float(n_mine), float(R_mine)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(red[0])
    n_total = int(tot[1])
    label = ("C5 synthetic DNase-seq: %d reads over %d sites +-%d bp, per-base" if which == "C5" else
             "C3 synthetic gene bodies (one sample): %d reads over %d genes +-%d bp, 50+150+50 bins")
    out = {"workload": (label + ", ONE problem sharded by region over %d GPU(s)") % (n_total, len(win), w["flank"][0],
                                                                                    world),
           "scaling": "strong", "n_gpus": world, "steps": steps,
           "ms_per_step": ms, "reads_per_s": n_total / (ms * 1e-3),
           "ms_device_resident": float(red[1]) + float(red[2]),
           "reads_per_s_device_resident": n_total / ((float(red[1]) + float(red[2])) * 1e-3),
           "phases_ms_max_over_ranks": {"exchange_reads (classify + NCCL all-to-all)": float(red[1]),
                                        "load + coverage + per-base matrix": float(red[2]),
                                        "matrix block D2H (own PCIe link)": float(red[3])},
           "reads_after_exchange": int(tot[2]), "regions": int(tot[3]), "matrix_cols": ncols,
           "matrix_bytes_total": int(tot[3]) * ncols * 8,
           "coverage_path_used": prob.stats.get("path"), "checksum": float(tot[0]),
           "stage_ms_rank0": {k: v[0] * v[1] / steps for k, v in stage.items()},
           "generation_s_this_rank": round(t_gen, 1)}
    return out


DUMP_BYTES = 64 << 20


def matrix_to_host(mat):
    """A device matrix [bins, regions] (column-major regions x bins, as the step writes it) as the
    regions x bins float64 array a caller receives.  Above DUMP_BYTES only whole rows are kept: a
    sample fixed by its seed and the row count, in row order, so every build keeps the same rows."""
    import torch
    ncols, n_rows = mat.shape
    if n_rows * ncols * 8 > DUMP_BYTES:
        rows = np.random.default_rng(0).choice(n_rows, size=max(DUMP_BYTES // (8 * ncols), 1), replace=False)
        mat = mat.index_select(1, torch.from_numpy(np.sort(rows)).to(mat.device))
    return mat.t().contiguous().cpu().numpy()


def bind_cpu_near_gpu(local):
    """One process per GPU: run this process (and place its page-locked buffers, by first touch)
    on the CPUs of the GPU's own NUMA node, so that the N uploads of a step do not cross the socket
    interconnect.  NVML knows the ideal CPU set of a device.  RCP_BENCH_BIND_CPU=0 turns it off."""
    if os.environ.get("RCP_BENCH_BIND_CPU", "1") == "0":
        return "off"
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        p = torch.cuda.get_device_properties(local)
        bus = "%08X:%02X:%02X.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return "nvml ideal CPUs of %s: %d of %d" % (bus, len(os.sched_getaffinity(0)), before)
    except Exception as e:       # no NVML, restricted cpuset, old torch: run unbound
        return "unbound (%s: %s)" % (type(e).__name__, str(e)[:60])


def run_b200(args):
    import torch
    import torch.distributed as dist

    import recoup_b200 as rb
    from recoup_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    cpu_binding = bind_cpu_near_gpu(local) if world > 1 else "one GPU: not bound"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # a mismatched collective must fail in minutes, not hang the box until the watchdog
        dist.init_process_group("nccl", device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(seconds=180))
    rb.init(local)
    rb.set_coverage_path(args.path)
    L = _lib.lib
    _lib.check(L.rcp_set_deferred_validation(1))
    dev = torch.device("cuda", local)
    stream = torch.cuda.ExternalStream(L.rcp_stream(), device=dev)
    env = {"rb": rb, "_lib": _lib, "L": L, "dev": dev, "stream": stream}
    peak, peak_src = peaks()

    # ---- this rank's headline problem: a full-size sample of the named workload (N > 1: an
    # independent replica per rank, weak scaling) ----
    w = W.CONFIGS[args.workload](scale=args.scale, seed=SEEDS[args.workload] + 7919 * rank)
    if args.read_order == "coordinate":
        order = np.lexsort((w["read_start"], w["read_chrom"]))
        for key in ("read_chrom", "read_start", "read_end", "read_strand"):
            w[key] = np.ascontiguousarray(w[key][order])
        del order
        w["name"] += " (reads coordinate-sorted)"
    prob = Problem(env, w)
    N, R = prob.N, prob.R
    is_rna = prob.is_rna

    # ---- N > 1: NCCL gather of the row blocks to rank 0 (the reference's do.call(rbind, ...)) on
    # its own stream; the output matrix is double buffered, so the gather of step k runs beside
    # the kernels of step k + 1.  The NCCL call is issued by a helper thread (the host is on the
    # critical path of a step; ctypes releases the GIL inside the library).
    prob.step()                                             # sizes the matrix
    ncols = prob.ncols
    bufs = [prob.out] + ([torch.empty_like(prob.out)] if world > 1 else [])
    gstream = torch.cuda.Stream(device=dev) if world > 1 else None
    gdone = [None, None]
    gather_box = {}
    gq = queue.Queue()
    gissued = [threading.Event(), threading.Event()]
    for e in gissued:
        e.set()
    gfail = []

    if world > 1 and args.exchange == "ce":
        from recoup_b200.sharding import PeerMatrix
        # rank 0's matrix (double buffered like the blocks), mapped into every rank of the box
        gather_box["peer"] = [PeerMatrix(R * world, ncols, dev, dst=0) for _ in range(2)]

    def gather_issue(k, ready):
        from recoup_b200.sharding import RowGather
        gstream.wait_event(ready)
        with torch.cuda.stream(gstream):
            if args.exchange == "ce":
                pm = gather_box["peer"][k % 2]
                pm.put(bufs[k % 2], rank * R, stream=gstream)     # copy engine, straight into place
                pm.fence()                                          # one-word all-reduce on gstream
                if rank == 0:
                    gather_box["full"] = pm.as_tensor()
            else:
                if "g" not in gather_box:       # buffers and row indices are set up once
                    gather_box["g"] = RowGather(ncols, np.arange(rank * R, (rank + 1) * R), R * world, dev,
                                                bufs[0].dtype, dst=0, sizes=[R] * world)
                gather_box["full"] = gather_box["g"].gather(bufs[k % 2])
            done = torch.cuda.Event()
            done.record(gstream)
        return done

    def gather_worker():
        torch.cuda.set_device(dev)
        while True:
            item = gq.get()
            if item is None:
                return
            k, ready = item
            try:
                gdone[k % 2] = gather_issue(k, ready)
            except BaseException as exc:    # never leave the main thread waiting for this gather
                gfail.append(exc)
            finally:
                gissued[k % 2].set()

    gthread = None
    if world > 1:
        gthread = threading.Thread(target=gather_worker, daemon=True)
        gthread.start()

    def gather_drain():
        for e in gissued:
            e.wait()
        if gfail:
            raise gfail[0]

    def full_step(k):
        buf = bufs[k % len(bufs)]
        if world > 1:
            gissued[k % 2].wait()           # the helper thread has issued the gather two steps back
            if gfail:
                raise gfail[0]
            if gdone[k % 2] is not None:
                stream.wait_event(gdone[k % 2])     # ... and it has read this buffer
        prob.step(out_ptr=buf.data_ptr(), ld=R)
        if world > 1:
            ready = torch.cuda.Event()
            ready.record(stream)            # the bin kernel of this step (library stream)
            gissued[k % 2].clear()
            gq.put((k, ready))

    def barrier():
        gather_drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ----
    sampler = ClockSampler(local)
    sampler.start()
    for k in range(max(args.warmup, 3)):
        full_step(k)
    barrier()

    # ---- timed: device-resident ----
    L.rcp_launch_count(1)
    _lib.check(L.rcp_timing_enable(1))
    _lib.check(L.rcp_timing_read(1, 0, None, None))
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    ev0.record(stream)
    for k in range(args.steps):
        full_step(k)
    if world > 1:
        gather_drain()
        for ev in gdone:                    # the timed region ends when the last gathers have landed
            if ev is not None:
                stream.wait_event(ev)
    ev1.record(stream)
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = int(L.rcp_launch_count(0))
    stage = stage_table(L, _lib)
    _lib.check(L.rcp_timing_enable(0))
    # taken here: the untimed steps below write the same buffers again
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = matrix_to_host(gather_box["full"] if world > 1 else bufs[(args.steps - 1) % len(bufs)])
    # The timed region is a few tens of milliseconds, shorter than one nvidia-smi period: keep
    # the same steps running (untimed) for about a second so that the clock record is taken UNDER
    # THIS LOAD.  The number of extra steps is agreed by all ranks (never a rank-local wall
    # clock around a collective).
    n_probe = torch.tensor([max(1, min(4000, int(1000.0 / max(elapsed_ms / args.steps, 1e-3))))],
                           dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(n_probe, op=dist.ReduceOp.MIN)
    n_probe = int(n_probe.item())
    for k in range(args.steps, args.steps + n_probe):
        full_step(k)
    barrier()
    clocks = sampler.stop(t_begin, time.time(), "timed region + ~1 s of the same steps (untimed)")

    # ---- N > 1: the exchanged matrix on rank 0 must hold every rank's rows ----
    exchange_ok = None
    if world > 1:
        k_last = args.steps + n_probe - 1
        mine = bufs[k_last % 2].double().sum().reshape(1)
        sums = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(sums, mine)
        if rank == 0:
            full = gather_box["full"]
            exchange_ok = True
            for r in range(world):
                got = float(full[:, r * R:(r + 1) * R].sum())
                want = float(sums[r])
                if not (abs(got - want) <= 1e-9 * max(abs(want), 1.0)) or want == 0.0:
                    exchange_ok = False
        gq.put(None)
        gthread.join()
        barrier()
        for pm in gather_box.get("peer", []):
            pm.close()
        gather_box.clear()
        barrier()

    # ---- the fused entry point (coverage not materialised), same problem ----
    fused = None
    if not is_rna and prob.equal_lengths and prob.bp["regionBinSize"] > 0:
        prob.out = bufs[0]
        prob.step()
        want = prob.out.clone()
        ms_f, stage_f = time_problem(env, prob, args.steps, 3, step_fn=prob.fused_step)
        same = bool(torch.equal(want, prob.out))
        del want
        fused = {"ms_per_step": ms_f, "reads_per_s": N / (ms_f * 1e-3), "matrix_equals_two_stage": same,
                 "algorithmic_bytes": 8 * N + 16 * R + 8 * R * ncols,
                 "stage_ms": {k: v[0] * v[1] / args.steps for k, v in stage_f.items()}}
        fused["frac_of_hbm_peak"] = fused["algorithmic_bytes"] / (ms_f * 1e-3) / 1e9 / peak

    # ---- timed: end to end through the public host API (pinned host buffers) ----
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a[:1]).dtype, pin_memory=True)
        t.numpy()[...] = a
        return t

    pins = [pinned(w[k]) for k in ("read_chrom", "read_start", "read_end", "read_strand")]
    host_views = [p.numpy() for p in pins]
    h2d = sum(v.nbytes for v in host_views)
    if is_rna:
        grl = rb.GRangesList(rb.GRanges(w["exon_chrom"], w["exon_start"], w["exon_end"],
                                        strand=w["exon_strand"], seqlevels=w["chrom_names"]),
                             w["exon_ptr"])
        h2d += sum(prob.ex[i].nbytes for i in range(4)) + 2 * 13 * R
    else:
        h2d += 13 * R
    d2h = 8 * R * ncols + 4 * R
    e2e_steps = max(2, min(args.steps, 5))
    phases = {"upload+map": 0.0, "coverage": 0.0, "profile+download": 0.0}
    clen = prob.clen
    widths_equal = bool(np.all(w["read_end"] - w["read_start"] == w["read_end"][0] - w["read_start"][0]))
    read_w = int(w["read_end"][0] - w["read_start"][0] + 1)
    e2e_in = {"seqnames": host_views[0], "views": host_views, "width": None}

    def e2e_step():
        """The calls a user of the reference API makes, on pinned HOST arrays."""
        t_a = time.perf_counter()
        hv = e2e_in["views"]
        if e2e_in["width"] is None:
            reads = rb.GRanges(e2e_in["seqnames"], hv[1], hv[2], strand=hv[3],
                               seqlevels=w["chrom_names"], seqlengths=clen)
        else:       # fixed-length library: an IRanges of ONE width, no end array anywhere
            reads = rb.GRanges(e2e_in["seqnames"], hv[1], width=e2e_in["width"], strand=hv[3],
                               seqlevels=w["chrom_names"], seqlengths=clen)
        sample = [dict(id="s", name="s", ranges=reads)]
        rb.device_reads(reads, w["frag_len"])
        t_b = time.perf_counter()
        if is_rna:
            rb.coverageRnaRef(sample, grl, prob.genes, w["flank"])
        else:
            if w["frag_len"]:
                sample[0]["coverage"] = rb.calcCoverage(reads, prob.win, frag_len=w["frag_len"])
            else:
                rb.coverageRef(sample, prob.genes, w["region"], w["flank"])
        t_c = time.perf_counter()
        rb.profileMatrix(sample, w["flank"], prob.bp)
        m = sample[0]["profile"]
        t_d = time.perf_counter()
        sample[0]["coverage"].free()
        for dr in reads._device.values():
            dr.free()
        reads._device.clear()
        phases["upload+map"] += t_b - t_a
        phases["coverage"] += t_c - t_b
        phases["profile+download"] += t_d - t_c
        return m

    def e2e_time(want_sum=None):
        # warm-up: two results alive at once, so that the library's pinned-buffer pool holds the
        # two output matrices the timed loop alternates between (page-locking 32 MB costs ~12 ms)
        keep = [e2e_step(), e2e_step()]
        if want_sum is not None:
            assert abs(float(keep[0].sum()) - want_sum) <= 1e-9 * max(abs(want_sum), 1.0)
        del keep
        for k in phases:
            phases[k] = 0.0
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            mat = e2e_step()
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / e2e_steps
        assert mat.shape == (R, ncols)
        return sec, dict(phases), float(mat.sum())

    # (1) dense arrays, reads in random order: seqnames, start, end int32 + strand int8 (13 B/read)
    e2e_dense_s, dense_phases, want_sum = e2e_time()
    h2d_dense = h2d

    # (2) the same reads grouped by chromosome as a coordinate-sorted BAM delivers them (random
    # order inside a chromosome: nothing on the device assumes an order).  A GRanges holds such
    # seqnames as ~25 runs (Rle), and rcp_reads_load_rle sends the runs instead of 4 bytes per read.
    order = np.argsort(host_views[0].astype(np.uint8), kind="stable")
    for p in pins:
        p.numpy()[...] = p.numpy()[order]
    del order
    seq_rle = rb.Rle.encode(host_views[0])
    e2e_in["seqnames"] = seq_rle
    h2d_bam = h2d - host_views[0].nbytes + 8 * seq_rle.nrun
    e2e_bam_s, bam_phases, _ = e2e_time(want_sum)
    n_runs = seq_rle.nrun

    # (3) ... and, for a fixed-length library, the ranges as the IRanges of ONE width they are:
    # start + width (a number) + strand -- rcp_reads_load_width; the ends never exist on the host
    # side of PCIe.  This is the representation the headline `e2e` is quoted on when the workload
    # has one read length; otherwise (2).
    e2e_fixed_s, fixed_phases, h2d_fixed = None, None, None
    if widths_equal and not is_rna:
        e2e_in["width"] = read_w
        h2d_fixed = h2d_bam - host_views[2].nbytes
        e2e_fixed_s, fixed_phases, _ = e2e_time(want_sum)
    del pins, host_views, e2e_in
    if e2e_fixed_s is not None:
        e2e_s, phases, h2d = e2e_fixed_s, fixed_phases, h2d_fixed
        e2e_inputs = ("reads grouped by chromosome (BAM order) as the GRanges of a fixed-length library "
                      "holds them: seqnames Rle (%d runs), start int32, ONE width (%d), strand int8 "
                      "-- 5 B/read cross PCIe" % (n_runs, read_w))
    else:
        e2e_s, phases, h2d = e2e_bam_s, bam_phases, h2d_bam
        e2e_inputs = ("reads grouped by chromosome (BAM order): seqnames Rle (%d runs), start, end int32, "
                      "strand int8 -- 9 B/read cross PCIe" % n_runs)

    # ---- reduce over ranks (max time) ----
    t = torch.tensor([elapsed_ms, e2e_s * 1e3, e2e_bam_s * 1e3, e2e_dense_s * 1e3], dtype=torch.float64,
                     device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_ms, e2e_bam_ms, e2e_dense_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    ms_per_step = elapsed_ms / args.steps
    value = world * N / (ms_per_step * 1e-3)
    e2e_value = world * N / (e2e_ms * 1e-3)
    stats = prob.stats
    total_len = stats["total_len"]
    headline_name = w["name"]
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(w)

    # ---- the other configs (one GPU) and the region-sharded C5 ----
    prob = None
    bufs = None
    w = None
    torch.cuda.empty_cache()
    configs = None
    headline = args.workload == "C2" and args.scale == 1.0
    if world == 1 and args.configs == "all" and headline:
        cs = args.configs_scale
        note = None if cs == 1.0 else "scaled by %.3g" % cs
        configs = {"C1": run_c1(env)}
        # C3: 8 samples over the same 60k genes; each sample is one step (per-sample numbers)
        per = []
        for smp in range(8):
            w3 = W.gene_bodies(scale=cs, seed=SEEDS["C3"])
            if smp:     # same genes, this sample's own reads
                w3.update({k: v for k, v in W.gene_bodies(scale=cs, seed=SEEDS["C3"] + 101 * smp).items()
                           if k.startswith("read_")})
            per.append(config_entry(env, w3, max(2, min(args.steps, 3)), peak, samples=8, note=note))
            del w3
        c3 = dict(per[0])
        c3["ms_per_sample"] = float(np.mean([e["ms_per_sample"] for e in per]))
        c3["ms_all_8_samples"] = float(np.sum([e["ms_per_sample"] for e in per]))
        c3["reads_per_s"] = float(np.sum([e["reads_per_sample"] for e in per]) / (c3["ms_all_8_samples"] * 1e-3))
        c3["per_sample_ms"] = [e["ms_per_sample"] for e in per]
        configs["C3"] = c3
        w4 = W.rnaseq(scale=cs)
        configs["C4"] = config_entry(env, w4, max(2, min(args.steps, 3)), peak, note=note)
        del w4
        torch.cuda.empty_cache()
        configs["import"] = run_import(env, 2_000_000)
        torch.cuda.empty_cache()
    strong = strong_c3 = None
    if args.strong == "on" and headline:
        strong = run_strong(env, args, world, rank)
        torch.cuda.empty_cache()
        strong_c3 = run_strong(env, args, world, rank, "C3")
        torch.cuda.empty_cache()
        if configs is not None:
            configs["C5"] = dict(strong, note="run through the region-sharded code path at W = 1; the matrix "
                                              "block download (8 GB D2H) is inside ms_per_step")

    if rank == 0:
        # Algorithmic bytes per KERNEL (the `roofline` object, dominant own kernel of the step): the
        # bytes that kernel cannot avoid moving -- a pass over the reads 8 B/read, the tile kernels
        # 4 B/covered base written + the candidates read once, the bin kernel 4 B/covered base +
        # 8 B/cell, the sort 8 B/key.
        cand = stats.get("candidates", 0)
        alg_kernel = {
            "blk_filter": 8 * N, "blk_scatter": 16 * cand, "blk_tile": 4 * total_len + 8 * cand,
            "blk_small": 4 * total_len + 8 * cand,
            "sp_split": 8 * N, "sp_sort": 8 * cand, "sp_tile": 4 * total_len + 4 * cand,
            "index_map": 22 * N, "index_sort": 8 * N,
            "cov_tile": 8 * N + 4 * total_len + 16 * R, "cov_small": 8 * N + 4 * total_len + 16 * R,
            "bkt_count": 8 * N, "bkt_scatter": 8 * N, "bkt_tile": 4 * total_len, "bkt_small": 4 * total_len,
            "prof_bin": 4 * total_len + 8 * R * ncols, "prof_base": 4 * total_len + 8 * R * ncols,
        }
        stage_roof, per_step = stage_roofline(stage, args.steps, N, R, ncols, total_len, peak)
        # measured DRAM traffic per launch (ncu --set full of this round's kernels), keyed by stage
        # (a figure is used only while the source file of its kernel still has the hash recorded
        # with the capture -- tools/make_traffic.py; a stale file reads as null, never as a number)
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "r02_traffic_C2.json")
        if headline and os.path.exists(tpath):
            import hashlib
            tj = json.load(open(tpath))
            for stage_name, fname in tj.get("file_of", {}).items():
                src = os.path.join(ROOT, "recoup_b200", "csrc", fname)
                if (stage_name in tj and os.path.exists(src) and
                        hashlib.sha256(open(src, "rb").read()).hexdigest() == tj["source_hash"].get(fname)):
                    traffic[stage_name] = tj[stage_name]
        own = {k: v for k, v in stage.items() if k in alg_kernel}
        dom = max(own, key=lambda k: own[k][0] * own[k][1]) if own else None
        roof = None
        if dom:
            per_launch_ms = own[dom][0]         # average over the launches of the timed region
            ach = alg_kernel[dom] / (per_launch_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": traffic.get(dom), "peak_source": peak_src,
                    "ms_per_step": per_step[dom], "ms_per_launch": per_launch_ms,
                    "launches_per_step": own[dom][1] / args.steps,
                    "algorithmic_bytes": alg_kernel[dom],
                    "kernels": {k: {"ms_per_launch": own[k][0], "launches_per_step": own[k][1] / args.steps,
                                    "algorithmic_bytes": alg_kernel[k],
                                    "frac": alg_kernel[k] / (own[k][0] * 1e-3) / 1e9 / peak}
                                for k in own},
                    "stages": stage_roof}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32 coverage / f64 matrix",
            "data": "synthetic",
            "config": {"workload": headline_name, "regions_per_gpu": R, "reads_per_gpu": N,
                       "matrix_cols": ncols, "covered_bases_per_gpu": total_len,
                       "null_regions": stats["n_null"],
                       "l2": "inputs (%.0f MB) and coverage (%.0f MB) exceed the 126 MB L2"
                             % (13 * N / 1e6, 4 * total_len / 1e6),
                       "coverage_path": args.path, "coverage_path_used": stats.get("path"),
                       "candidates_per_gpu": stats.get("candidates"),
                       "parallelism": ("one GPU" if world == 1 else
                                       "%d independent replicas of the workload, one per GPU (weak scaling; "
                                       "every rank its own reads and regions), row blocks %s on a second "
                                       "stream; the ONE-problem region-sharded run is in `strong`"
                                       % (world, "put straight into rank 0's matrix by the copy engine over "
                                                 "NVLink (CUDA IPC mapping), fenced by a one-word NCCL all-reduce"
                                          if args.exchange == "ce" else
                                          "gathered to rank 0 with NCCL (dist.gather + placement)"))},
            "stage_ms_per_step": per_step,
            "region_bins_per_s": world * R * ncols / (ms_per_step * 1e-3),
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "phases_ms": {k: 1e3 * v / e2e_steps for k, v in phases.items()},
                    "inputs": e2e_inputs},
            "e2e_bam_order": {"value": world * N / (e2e_bam_ms * 1e-3), "unit": UNIT,
                              "h2d_bytes_per_step": int(h2d_bam), "d2h_bytes_per_step": int(d2h),
                              "ms_per_step": e2e_bam_ms, "steps": e2e_steps,
                              "phases_ms": {k: 1e3 * v / e2e_steps for k, v in bam_phases.items()},
                              "inputs": "the same reads with the end array as well (general GRanges): "
                                        "seqnames Rle (%d runs), start, end int32 + strand int8" % n_runs},
            "e2e_dense_arrays": {"value": world * N / (e2e_dense_ms * 1e-3), "unit": UNIT,
                                 "h2d_bytes_per_step": int(h2d_dense), "d2h_bytes_per_step": int(d2h),
                                 "ms_per_step": e2e_dense_ms, "steps": e2e_steps,
                                 "phases_ms": {k: 1e3 * v / e2e_steps for k, v in dense_phases.items()},
                                 "inputs": "reads in random order as four dense arrays (round 1's `e2e`): "
                                           "seqnames, start, end int32 + strand int8 -- 13 B/read"},
            "gpu_launches": launches, "clocks": clocks,
        }
        if fused is not None:
            out["fused"] = fused
        if configs is not None:
            out["configs"] = configs
        out["cpu_binding_rank0"] = cpu_binding
        if strong is not None:
            out["strong"] = strong
        if strong_c3 is not None:
            out["strong_C3"] = strong_c3
        if exchange_ok is not None:
            out["exchange_verified"] = exchange_ok
        if cpu is not None:
            out["cpu_baseline"] = cpu
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "profile.npy"), dumped)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
