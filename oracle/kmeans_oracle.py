"""ORACLE (test infrastructure, never imported by the product): `set.seed(seed); kmeans(x, k,
iter.max, nstart, algorithm)` as stats::kmeans runs it for kmeansDesign (util.R:140-197).
Parity unpinned: R's sources are not vendored; this restates its documented sequence.

* The draws, one RNG stream (`oracle/r_rng.py`): nstart == 1: `x[sample.int(m, k), ]`; when those
  rows hold a duplicate, or nstart >= 2: `cn <- unique(x)`, then `cn[sample.int(nrow(cn), k), ]`
  for the first start and one more `sample.int(nrow(cn), k)` per further start.
* `unique(x)`: distinct rows in first-occurrence order, compared exactly with -0.0 == 0.0 (R
  compares `paste(row, collapse = "\\r")`, 15 significant digits: rows that differ only beyond
  that are duplicates to R and distinct here; DESIGN.md section 2).
* The starts run through `oracle/kmeans_oracle.c` (kmeans_Lloyd, kmeans_MacQueen and AS 136,
  built with -ffp-contract=off), and the first start with the strictly smallest sum(wss) is kept.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .r_rng import RRandom

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle_kmeans.so")

ALGORITHMS = {"Hartigan-Wong": 1, "Lloyd": 2, "Forgy": 2, "MacQueen": 3}
_SRC = os.path.join(_HERE, "kmeans_oracle.c")
# /usr/bin/gcc is named explicitly when present, as in oracle/Makefile
_GCC = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
_lib = None


def _compile(out):
    # -ffp-contract=off: no product is fused into an add, as in x86-64 builds of R
    subprocess.check_call([_GCC, "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", out,
                           _SRC])


def build(force=False):
    """Compiles kmeans_oracle.c next to it when missing or stale; a read-only tree gets the
    library in a per-user temporary directory instead.  Returns its path."""
    if not force and os.path.exists(_SO) and os.path.getmtime(_SO) >= os.path.getmtime(_SRC):
        return _SO
    if os.access(_HERE, os.W_OK):
        _compile(_SO)
        return _SO
    out = os.path.join(tempfile.gettempdir(), "recoup_b200_oracle_kmeans_%d.so" % os.getuid())
    if force or not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(_SRC):
        _compile(out)
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, i64 = C.c_void_p, C.c_int64
        for name in ("okm_lloyd", "okm_macqueen"):
            getattr(L, name).argtypes = [vp, i64, i64, i64, vp, C.c_int, vp, vp, vp, vp]
        L.okm_hartigan_wong.argtypes = [vp, i64, i64, i64, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                        vp, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def unique_rows(x):
    """0-based indices of the distinct rows of x in first-occurrence order (-0.0 == 0.0)."""
    x = np.asarray(x, dtype=np.float64) + 0.0          # -0.0 + 0.0 = +0.0
    seen = set()
    out = []
    for i in range(x.shape[0]):
        key = x[i].tobytes()
        if key not in seen:
            seen.add(key)
            out.append(i)
    return np.array(out, dtype=np.int64)


class KmeansError(ValueError):
    pass


def initial_centres(x, k, nstart, seed=42, sample_kind="Rejection"):
    """The row indices (0-based, one row of k per start) that kmeans takes as initial centres."""
    x = np.asarray(x, dtype=np.float64)
    m = x.shape[0]
    rng = RRandom(seed, sample_kind)
    use_unique = nstart >= 2
    if nstart == 1:
        rows = np.array(rng.sample_int(m, k), dtype=np.int64) - 1
        c = x[rows] + 0.0
        use_unique = len({r.tobytes() for r in c}) < k
        if not use_unique:
            return rows[None, :]
    cn = unique_rows(x)
    if cn.shape[0] < k:
        raise KmeansError("more cluster centers than distinct data points.")
    return np.stack([cn[np.array(rng.sample_int(cn.shape[0], k), dtype=np.int64) - 1] for _ in range(nstart)])


def run_start(x, centres, algorithm, iter_max):
    """One start (do_one): dict(cluster 1-based, centers k x p, withinss, size, iter, ifault)."""
    x = np.asfortranarray(x, dtype=np.float64)
    m, p = x.shape
    k = centres.shape[0]
    cen = np.asfortranarray(centres, dtype=np.float64).copy(order="F")
    cl = np.zeros(m, dtype=np.int32)
    nc = np.zeros(k, dtype=np.int32)
    wss = np.zeros(k, dtype=np.float64)
    it = C.c_int(iter_max)
    ifault = C.c_int(0)
    L = lib()
    meth = ALGORITHMS[algorithm]
    if k == 1:
        meth = 3
    ld = max(m, 1)
    if meth == 1:
        work = dict(ic2=np.zeros(m, np.int32), d=np.zeros(m), an1=np.zeros(k), an2=np.zeros(k),
                    itran=np.zeros(k, np.int32), ncp=np.zeros(k, np.int64), live=np.zeros(k, np.int64))
        L.okm_hartigan_wong(_p(x), m, p, ld, _p(cen), k, _p(cl), C.byref(it), _p(nc), _p(wss), C.byref(ifault),
                            *[_p(work[n]) for n in ("ic2", "d", "an1", "an2", "itran", "ncp", "live")])
        if ifault.value == 1:
            raise KmeansError("empty cluster: try a better set of initial centers")
        if ifault.value == 3:
            raise KmeansError("number of cluster centres must lie between 1 and nrow(x)")
    else:
        (L.okm_lloyd if meth == 2 else L.okm_macqueen)(_p(x), m, p, ld, _p(cen), k, _p(cl), C.byref(it), _p(nc),
                                                       _p(wss))
        if it.value > iter_max:
            ifault.value = 2
    return dict(cluster=cl, centers=cen, withinss=wss, size=nc, iter=it.value, ifault=ifault.value)


def kmeans(x, k, iter_max=10, nstart=1, algorithm="Hartigan-Wong", seed=42, sample_kind="Rejection",
           all_starts=False):
    """The kmeans() result as a dict; all_starts=True also returns every start's result and the
    index of the chosen one."""
    x = np.asarray(x, dtype=np.float64)
    if not np.all(np.isfinite(x)):
        raise KmeansError("NA/NaN/Inf in foreign function call (arg 1)")
    rows = initial_centres(x, k, nstart, seed, sample_kind)
    starts = [run_start(x, x[r], algorithm, iter_max) for r in rows]
    best = 0
    tots = [float(np.sum(np.asarray(s["withinss"], dtype=np.longdouble))) for s in starts]
    for s in range(1, len(starts)):
        if tots[s] < tots[best]:
            best = s
    z = dict(starts[best])
    xc = x - x.mean(axis=0)
    z["totss"] = float(np.sum(xc * xc))
    z["tot_withinss"] = tots[best]
    z["betweenss"] = z["totss"] - tots[best]
    if all_starts:
        z["starts"] = starts
        z["best"] = best
        z["tots"] = tots
    return z
