"""rcp_kmeans on the device against the C restatement of stats::kmeans on one CPU core.

k = 5, nstart = 20, iter.max = 20, every algorithm, on seeded clustered matrices of the project's
shapes: C2 (2e4 x 400), C3 (6e4 x 2000), C5 (1e6 x 1000).  The matrix is generated on the device
(torch, seeded) and passed device-resident (RCP_MEM_DEVICE).  Per line: the median of --reps
calls timed with a host clock around the synchronised call, iter, and -- from a separate
torch.profiler run -- the share of kernel time in the one-CTA-per-start walker (MacQueen,
Hartigan-Wong).  The CPU line is oracle/kmeans_oracle.c ("CPU restatement, not R") on one core:
starts are run one after the other until --cpu-budget seconds are spent; the 20-start time is
measured when they all fit, else extrapolated from the starts that ran (at least one; marked so);
matrices above --cpu-max-cells get no CPU line, and the line says so.  Writes one JSON file with
the card name and power limit read in the same run, after every line.

    python tools/bench_kmeans.py --shapes C2,C3,C5 --out profiles/kmeans_b200.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"C2": (20_000, 400), "C3": (60_000, 2_000), "C5": (1_000_000, 1_000)}
ALGS = {"Hartigan-Wong": 1, "Lloyd": 2, "MacQueen": 3}
K, NSTART, ITER_MAX = 5, 20, 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim = [s.strip() for s in q.split(",")]
        return name, plim
    except Exception as e:   # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def matrix(torch, m, p, seed):
    """K Gaussian blobs (sd 1, centres sd 3 apart) plus 10 % zero rows, column-major fp64 on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.randn(K, p, generator=g, device="cuda", dtype=torch.float64) * 3.0
    lab = torch.randint(0, K, (m,), generator=g, device="cuda")
    xt = torch.empty((p, m), dtype=torch.float64, device="cuda")        # x^T row-major = x column-major
    step = max(1, (1 << 27) // p)
    for a in range(0, m, step):
        b = min(m, a + step)
        blk = cen[lab[a:b]] + torch.randn(b - a, p, generator=g, device="cuda", dtype=torch.float64)
        xt[:, a:b] = blk.T
    zero = torch.rand(m, generator=g, device="cuda") < 0.1
    xt[:, zero] = 0.0
    return xt


def run_device(lib, torch, xt, m, p, alg):
    cl = torch.empty(m, dtype=torch.int32, device="cuda")
    cen = torch.empty(K * p, dtype=torch.float64, device="cuda")
    wss = torch.empty(K, dtype=torch.float64, device="cuda")
    size = torch.empty(K, dtype=torch.int32, device="cuda")
    tot, it, fault, warn = C.c_double(), C.c_int(), C.c_int(), C.c_int()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rc = lib.rcp_kmeans(C.c_void_p(xt.data_ptr()), m, p, m, K, NSTART, ITER_MAX, ALGS[alg], 42, 0, 1,
                        C.c_void_p(cl.data_ptr()), C.c_void_p(cen.data_ptr()), C.c_void_p(wss.data_ptr()),
                        C.c_void_p(size.data_ptr()), C.byref(tot), C.byref(it), C.byref(fault), C.byref(warn))
    lib.rcp_sync()
    dt = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError(lib.rcp_last_error().decode())
    return dt, dict(iter=it.value, ifault=fault.value, warnings=warn.value, size=size.cpu().tolist(),
                    tot_withinss=float(wss.sum().item()))


def walker_share(lib, torch, xt, m, p, alg):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_device(lib, torch, xt, m, p, alg)
    tot = walk = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if "km_" in e.key:
            tot += t
            if "km_walk_kernel" in e.key:
                walk += t
    return (walk / tot) if tot > 0 else None, tot / 1e3


def run_cpu(x, alg, budget):
    from oracle import kmeans_oracle as O
    rows = O.initial_centres(x, K, NSTART, 42)
    done, t0 = 0, time.perf_counter()
    iters = []
    for r in rows:
        if done and time.perf_counter() - t0 > budget:
            break
        iters.append(O.run_start(x, x[r], alg, ITER_MAX)["iter"])
        done += 1
        if time.perf_counter() - t0 > budget and done == 1 and budget > 0:
            break
    dt = time.perf_counter() - t0
    return dict(starts_run=done, seconds_run=round(dt, 3), per_start_s=round(dt / done, 4),
                nstart20_s=round(dt / done * NSTART, 3), extrapolated=done < NSTART, iters=iters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C2,C3,C5")
    ap.add_argument("--algorithms", default=",".join(ALGS), help="in this order")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls per line first (0: for C5's long calls)")
    ap.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of CPU restatement per line")
    ap.add_argument("--cpu-max-cells", type=float, default=2.5e8,
                    help="no CPU line above this many matrix cells (the host copy alone would dominate)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("no GPU: this tool measures on the device")
    import recoup_b200 as rb
    from recoup_b200 import _lib
    rb.init(0)
    lib = _lib.lib
    name, plim = card()
    res = dict(tool="tools/bench_kmeans.py", gpu=name, power_limit=plim, k=K, nstart=NSTART, iter_max=ITER_MAX,
               timing="host clock around the synchronised call, median of reps; device-resident input", lines=[])
    for shape in args.shapes.split(","):
        m, p = SHAPES[shape]
        xt = matrix(torch, m, p, 7)
        x_host = None
        for alg in args.algorithms.split(","):
            for _ in range(args.warmup):                          # module load, first allocations
                run_device(lib, torch, xt, m, p, alg)
            times, info = [], None
            for _ in range(args.reps):
                dt, info = run_device(lib, torch, xt, m, p, alg)
                times.append(dt)
            share, ktime = walker_share(lib, torch, xt, m, p, alg)
            line = dict(shape=shape, m=m, p=p, algorithm=alg, gpu_s=round(float(np.median(times)), 4),
                        gpu_s_all=[round(t, 4) for t in times], kernel_ms_profiled=round(ktime, 2),
                        walker_share=None if share is None or alg == "Lloyd" else round(share, 3), **info)
            if m * p <= args.cpu_max_cells:
                if x_host is None:
                    x_host = np.asfortranarray(xt.T.cpu().numpy())
                cpu = run_cpu(x_host, alg, args.cpu_budget)
                line["cpu_restatement_not_R"] = cpu
                line["speedup_vs_cpu_restatement"] = round(cpu["nstart20_s"] / line["gpu_s"], 1)
            else:
                line["cpu_restatement_not_R"] = "skipped: %d cells exceed the CPU line's limit of %.2g" % (
                    m * p, args.cpu_max_cells)
            res["lines"].append(line)
            print(json.dumps(line), flush=True)
            if args.out:                                          # after every line: long runs keep what they measured
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "w") as f:
                    json.dump(res, f, indent=1)
        del xt
        torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=name, power_limit=plim, lines=len(res["lines"]))))


if __name__ == "__main__":
    main()
