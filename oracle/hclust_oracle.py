"""ORACLE (test infrastructure, never imported by the product): `hclust(dist(x), "complete")` as
ComplexHeatmap clusters heat-map rows for orderBy$what = "hc<n>" / "hca".  Parity unpinned: R's
sources are not vendored; oracle/hclust_oracle.c restates R_euclidean, hclust.f (complete
linkage) and HCASS2 literally, built with -ffp-contract=off (oracle/cbuild.py).
"""
import ctypes as C

import numpy as np

from .cbuild import build_shared

_lib = None


class HclustError(ValueError):
    pass


def build(force=False):
    """Compiles hclust_oracle.c (with OpenMP where gcc has it) when missing or stale."""
    return build_shared("hclust_oracle", openmp=True, force=force)


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, i64 = C.c_void_p, C.c_int64
        L.ohc_dist.argtypes = [vp, i64, i64, i64, vp]
        L.ohc_dist.restype = None
        L.ohc_hclust.argtypes = [C.c_int, vp, vp, vp, vp, vp, vp, vp]
        L.ohc_hclust.restype = C.c_int
        L.ohc_hcass2.argtypes = [C.c_int, vp, vp, vp, vp, vp]
        L.ohc_hcass2.restype = None
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def dist(x):
    """dist(x) (Euclidean) as R stores it: the lower triangle by columns, n (n - 1) / 2 values."""
    x = np.asfortranarray(x, dtype=np.float64)
    n, p = x.shape
    d = np.empty(n * (n - 1) // 2, dtype=np.float64)
    lib().ohc_dist(_p(x), n, p, max(n, 1), _p(d))
    return d


def hclust_dist(d, n):
    """hclust(d, "complete") of a condensed distance vector (which is not modified): 1-based ia,
    ib and the heights, before HCASS2."""
    diss = np.array(d, dtype=np.float64)
    ia = np.zeros(n, np.int32)
    ib = np.zeros(n, np.int32)
    crit = np.zeros(n, np.float64)
    if lib().ohc_hclust(n, _p(diss), _p(ia), _p(ib), _p(crit), _p(np.zeros(n, np.int32)), _p(np.zeros(n)),
                        _p(np.zeros(n, np.int8))):
        raise HclustError("a distance reaches 1e300, hclust's INF")
    return ia[:n - 1], ib[:n - 1], crit[:n - 1]


def hcass2(n, ia, ib):
    """merge ((n - 1) x 2, R's signs) and order (1-based) from 1-based ia / ib."""
    a = np.zeros(n, np.int32)
    b = np.zeros(n, np.int32)
    a[:n - 1] = ia
    b[:n - 1] = ib
    order = np.zeros(n, np.int32)
    iia = np.zeros(n, np.int32)
    iib = np.zeros(n, np.int32)
    lib().ohc_hcass2(n, _p(a), _p(b), _p(order), _p(iia), _p(iib))
    return np.stack([iia[:n - 1], iib[:n - 1]], axis=1), order


def hclust(x):
    """hclust(dist(x), "complete"): dict(merge, height, order)."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim != 2:
        raise HclustError("x must be a matrix")
    n = x.shape[0]
    if n < 2:
        raise HclustError("must have n >= 2 objects to cluster")
    if not np.all(np.isfinite(x)):
        raise HclustError("NA/NaN/Inf in foreign function call (arg 1)")
    ia, ib, crit = hclust_dist(dist(x), n)
    merge, order = hcass2(n, ia, ib)
    return dict(merge=merge, height=crit, order=order)
