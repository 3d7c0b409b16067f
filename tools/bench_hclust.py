"""rcp_hclust (hclust(dist(x), "complete")) on the device against the C restatement on one CPU core.

Shapes: C1 (100 x 200), C2 (2e4 x 200), C3 (6e4 x 250) and R's limit (65 536 x 200), seeded
clustered profiles with 10 % zero rows (tools/bench_kmeans.py's generator), generated and passed
device-resident (RCP_MEM_DEVICE).  Per line:
  * the whole call: CUDA events around it, median of --reps after a warm-up call;
  * the distance kernel, the initial-NN pass and the merge loop: device time of each kernel from a
    separate torch.profiler run;
  * counts from the shapes: the distance kernel does 3 p n (n-1) / 2 fp64 operations and writes
    8 n^2 bytes; the merge loop reads rows I2 and J2 over the alive rows (8 n^2 bytes over all
    steps) and writes row and column I2 (8 n^2 bytes; the column's 8-byte stores move 32-byte
    sectors), rescans not counted -- so its bandwidth figure is a lower bound;
  * shares of the measured HBM figure (6 456 GB/s) and the merge loop's time per step.
The CPU line is oracle/hclust_oracle.c on one core ("CPU restatement, not R"): on the first n0 rows
of the same matrix, n0 the largest of --cpu-rows that fits --cpu-budget seconds, extrapolated to n
by (n / n0)^2 (both dist and the merge loop do O(n^2) work here) and marked so.  Writes one JSON
file with the card name and power limit read in the same run, after every line.

    python tools/bench_hclust.py --out profiles/hclust_b200.json
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

os.environ["OMP_NUM_THREADS"] = "1"          # the CPU line runs on one core

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SHAPES = {"C1": (100, 200), "C2": (20_000, 200), "C3": (60_000, 250), "L": (65_536, 200)}
HBM_GBS = 6456.0


def run_device(lib, torch, xt, n, p, out):
    merge, height, order = out
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    rc = lib.rcp_hclust(C.c_void_p(xt.data_ptr()), n, p, n, 3, 1, C.c_void_p(merge.data_ptr()),
                        C.c_void_p(height.data_ptr()), C.c_void_p(order.data_ptr()))
    e.record()
    torch.cuda.synchronize()
    if rc != 0:
        raise RuntimeError(lib.rcp_last_error().decode())
    return s.elapsed_time(e) / 1e3


def kernel_times(lib, torch, xt, n, p, out):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_device(lib, torch, xt, n, p, out)
    t = {"hc_dist_kernel": 0.0, "hc_nn_kernel": 0.0, "hc_merge_kernel": 0.0}
    for ev in prof.key_averages():
        dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        for k in t:
            if k in ev.key:
                t[k] += dt / 1e6
    return t


def run_cpu(x, n, rows, budget):
    from oracle import hclust_oracle as H
    best = None
    for n0 in sorted(set(min(n, r) for r in rows)):
        t0 = time.perf_counter()
        d = H.dist(x[:n0])
        t1 = time.perf_counter()
        H.hclust_dist(d, n0)
        t2 = time.perf_counter()
        del d
        best = (n0, t1 - t0, t2 - t1)
        if t2 - t0 > budget / 4 or n0 == n:
            break
    n0, td, tl = best
    f = (n / n0) ** 2
    return dict(rows_run=n0, dist_s_run=round(td, 3), loop_s_run=round(tl, 3), dist_s=round(td * f, 2),
                loop_s=round(tl * f, 2), total_s=round((td + tl) * f, 2), extrapolated=n0 < n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C1,C2,C3,L")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of CPU restatement per line")
    ap.add_argument("--cpu-rows", default="100,1000,2000,4000,8000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("no GPU: this tool measures on the device")
    import recoup_b200 as rb
    from bench_kmeans import card, matrix
    from recoup_b200 import _lib
    rb.init(0)
    lib = _lib.lib
    name, plim = card()
    res = dict(tool="tools/bench_hclust.py", gpu=name, power_limit=plim, hbm_gbs_measured=HBM_GBS,
               timing="CUDA events around the call, median of reps after one warm-up; kernel times from a "
                      "separate torch.profiler run; device-resident input", lines=[])
    rows = [int(r) for r in args.cpu_rows.split(",")]
    for shape in args.shapes.split(","):
        n, p = SHAPES[shape]
        xt = matrix(torch, n, p, 7)
        out = (torch.empty(2 * (n - 1), dtype=torch.int32, device="cuda"),
               torch.empty(n - 1, dtype=torch.float64, device="cuda"),
               torch.empty(n, dtype=torch.int32, device="cuda"))
        run_device(lib, torch, xt, n, p, out)
        times = [run_device(lib, torch, xt, n, p, out) for _ in range(args.reps)]
        kt = kernel_times(lib, torch, xt, n, p, out)
        call = float(np.median(times))
        dist_flop = 3.0 * p * n * (n - 1) / 2
        dist_bytes = 8.0 * n * n
        loop_bytes = 16.0 * n * n
        td, tl = kt["hc_dist_kernel"], kt["hc_merge_kernel"]
        line = dict(shape=shape, n=n, p=p, call_s=round(call, 4), call_s_all=[round(t, 4) for t in times],
                    dist_kernel_s=round(td, 5), nn_kernel_s=round(kt["hc_nn_kernel"], 5),
                    merge_loop_s=round(tl, 4), merge_us_per_step=round(tl / (n - 1) * 1e6, 3),
                    dist_tflops=round(dist_flop / td / 1e12, 2) if td else None,
                    dist_write_gbs=round(dist_bytes / td / 1e9, 1) if td else None,
                    dist_write_share_of_hbm=round(dist_bytes / td / 1e9 / HBM_GBS, 3) if td else None,
                    loop_gbs_lower_bound=round(loop_bytes / tl / 1e9, 1) if tl else None,
                    loop_share_of_hbm_lower_bound=round(loop_bytes / tl / 1e9 / HBM_GBS, 3) if tl else None,
                    height_max=float(out[1].max().item()))
        cpu = run_cpu(np.asfortranarray(xt.T.cpu().numpy()), n, rows, args.cpu_budget)
        line["cpu_restatement_not_R_one_core"] = cpu
        line["speedup_vs_cpu_restatement"] = round(cpu["total_s"] / call, 1)
        res["lines"].append(line)
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
        del xt, out
        torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=name, power_limit=plim, lines=len(res["lines"]))))


if __name__ == "__main__":
    main()
