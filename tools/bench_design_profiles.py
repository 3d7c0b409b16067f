"""rcp_matrix_group_col_profile (the curves of calcDesignPlotProfiles) on the device.

Shapes: C2 (2e4 x 200), C3 (6e4 x 250) and C5 (1e6 x 1 000), seeded gamma profiles with 20 % zero
rows, generated and passed device-resident (RCP_MEM_DEVICE).  Codes: G in {1, 5, 50} levels dealt
out interleaved, as k-means labels of unordered rows come.  Per line (shape, G, mean | median):
  * the call: CUDA events around it, median of --reps after one warm-up call;
  * kernel times and the number of kernel launches of one call, from a separate torch.profiler run;
  * the matrix bytes (8 n p) over the call time, and that rate as a share of the measured HBM
    figure (6 456 GB/s) -- the mean path reads the matrix twice and, for G > 1, copies it once;
  * the naive composition: for every level, index the level's rows into a new device matrix and
    call rcp_matrix_col_profile on it (CUDA events around all G of them, same repetitions).
Writes one JSON file with the card name and power limit read in the same run, after every line.

    python tools/bench_design_profiles.py --out profiles/design_profiles_b200.json
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SHAPES = {"C2": (20_000, 200), "C3": (60_000, 250), "C5": (1_000_000, 1_000)}
HBM_GBS = 6456.0


def matrix(torch, n, p, seed):
    """gamma(0.6, 3) cells, 20 % zero rows; x^T row-major = x column-major fp64 on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    xt = torch.empty((p, n), dtype=torch.float64, device="cuda")
    conc = torch.full((p,), 0.6, dtype=torch.float64, device="cuda")
    step = max(1, (1 << 27) // p)
    for a in range(0, n, step):
        b = min(n, a + step)
        xt[:, a:b] = torch.distributions.Gamma(conc, 1.0 / 3.0).sample((b - a,)).T
    xt[:, torch.rand(n, generator=g, device="cuda") < 0.2] = 0.0
    return xt


def codes_of(torch, n, G, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.arange(n, device="cuda", dtype=torch.int64) % G + 1
    return base[torch.randperm(n, generator=g, device="cuda")].to(torch.int32).contiguous()


def timed(torch, fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C2,C3,C5")
    ap.add_argument("--groups", default="1,5,50")
    ap.add_argument("--stats", default="mean,median")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("no GPU: this tool measures on the device")
    from torch.profiler import ProfilerActivity, profile

    import recoup_b200 as rb
    from bench_kmeans import card
    from recoup_b200 import _lib
    rb.init(0)
    lib = _lib.lib
    name, plim = card()
    res = dict(tool="tools/bench_design_profiles.py", gpu=name, power_limit=plim, hbm_gbs_measured=HBM_GBS,
               timing="CUDA events around the call, median of reps after one warm-up; kernel times and launch "
                      "counts from a separate torch.profiler run; device-resident input", lines=[])
    stat_code = {"mean": 0, "median": 1}
    for shape in args.shapes.split(","):
        torch.manual_seed(11)
        n, p = SHAPES[shape]
        xt = matrix(torch, n, p, 7)
        for G in [int(g) for g in args.groups.split(",")]:
            codes = codes_of(torch, n, G, 3)
            cen = torch.empty((p, G), dtype=torch.float64, device="cuda")
            spr = torch.empty_like(cen)
            level_rows = [torch.nonzero(codes == g + 1).squeeze(1) for g in range(G)]
            c1 = torch.empty(p, dtype=torch.float64, device="cuda")
            s1 = torch.empty_like(c1)
            for stat in args.stats.split(","):
                sc = stat_code[stat]

                def call():
                    rc = lib.rcp_matrix_group_col_profile(C.c_void_p(xt.data_ptr()), n, p, n,
                                                          C.c_void_p(codes.data_ptr()), G, sc, 0, _lib.MEM_DEVICE,
                                                          C.c_void_p(cen.data_ptr()), C.c_void_p(spr.data_ptr()))
                    if rc != 0:
                        raise RuntimeError(lib.rcp_last_error().decode())
                    _lib.check(lib.rcp_sync())

                def naive():
                    for g in range(G):
                        sub = xt.index_select(1, level_rows[g])           # the level's rows, column-major
                        torch.cuda.synchronize()
                        rc = lib.rcp_matrix_col_profile(C.c_void_p(sub.data_ptr()), sub.shape[1], p, sub.shape[1],
                                                        sc, 0, _lib.MEM_DEVICE, C.c_void_p(c1.data_ptr()),
                                                        C.c_void_p(s1.data_ptr()))
                        if rc != 0:
                            raise RuntimeError(lib.rcp_last_error().decode())
                        _lib.check(lib.rcp_sync())
                        cen[:, g].copy_(c1)
                        spr[:, g].copy_(s1)
                        del sub

                call()
                times = [timed(torch, call) for _ in range(args.reps)]
                want_c = cen.clone()
                naive()
                naive_times = [timed(torch, naive) for _ in range(args.reps)]
                same = bool(torch.equal(torch.nan_to_num(cen, 7.0), torch.nan_to_num(want_c, 7.0)))
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    call()
                kern, launches = {}, 0
                for ev in prof.key_averages():
                    if ev.device_type is not None and "cuda" in str(ev.device_type).lower():
                        if "Memcpy" in ev.key or "Memset" in ev.key:
                            continue
                        dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                        kern[ev.key[:80]] = round(dt / 1e6, 6)
                        launches += ev.count
                t = float(np.median(times))
                tn = float(np.median(naive_times))
                mb = 8.0 * n * p
                line = dict(shape=shape, n=n, p=p, G=G, stat=stat, call_s=round(t, 5),
                            call_s_all=[round(x, 5) for x in times], naive_s=round(tn, 5),
                            naive_s_all=[round(x, 5) for x in naive_times], speedup_vs_naive=round(tn / t, 2),
                            naive_center_equal=same, matrix_gb=round(mb / 1e9, 3),
                            matrix_gbs=round(mb / t / 1e9, 1), share_of_hbm=round(mb / t / 1e9 / HBM_GBS, 3),
                            kernel_launches=launches, kernel_s=round(sum(kern.values()), 5), kernels=kern)
                res["lines"].append(line)
                print(json.dumps({k: v for k, v in line.items() if k != "kernels"}), flush=True)
                if args.out:
                    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                    with open(args.out, "w") as f:
                        json.dump(res, f, indent=1)
            del cen, spr, codes, level_rows
            torch.cuda.empty_cache()
        del xt
        torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=name, power_limit=plim, lines=len(res["lines"]))))


if __name__ == "__main__":
    main()
