"""Host mirror of the reductions /root/reference/R/plot.R runs over finished `$profile` matrices,
over librecoup_b200.so (SURVEY 8f, N4):

    calcPlotProfiles(input, opts, ...)   average curve + band per sample        plot.R:949-990
    calcDesignPlotProfiles(input, design, opts)  the same per design level and sample
    orderProfiles(input, opts)           heat-map row order (sum / max / avg)   plot.R:1035-1150
    heatmapScale(input, ...)             upper colour limit from quantiles      plot.R:513-545
    kmeans(x, centers, ...)              stats::kmeans as kmeansDesign calls it
    kmeansDesign(input, design, kmParams) heat-map clusters as a design column  util.R:140-197
    hclust(x, method)                    stats::hclust(dist(x)) of heat-map rows
    heatmapClusters(input, opts, split)  the cluster_rows dendrograms of orderBy = "hc<n>" / "hca"

`opts` is the nested dict of the reference (`opts["plotParams"]["sumStat"]`, ...).  Matrices are
the `ProfileMatrix` objects profileMatrix() returns (host, column-major); they are staged to the
GPU by the library, so a device pointer can be passed through the C ABI directly instead
(`mem = RCP_MEM_DEVICE`) when the matrix never left the device.
"""
import ctypes as C
import re
import warnings

import numpy as np

from . import _lib

_ROW = {"sum": 0, "max": 1, "avg": 2}


def _f(mat):
    m = np.asfortranarray(mat, dtype=np.float64)
    if m.ndim != 2:
        raise ValueError("a profile must be a matrix")
    return m


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


def colProfile(mat, avgfun="mean", scale="natural"):
    """apply(x, 2, avgfun) and apply(x, 2, sd | mad), after log2(x + 1) for scale "log2"."""
    if avgfun not in ("mean", "median"):
        raise ValueError("sumStat must be mean or median")
    m = _f(mat)
    _lib.ensure_init()
    center = np.empty(m.shape[1], dtype=np.float64)
    spread = np.empty(m.shape[1], dtype=np.float64)
    _lib.check(_lib.lib.rcp_matrix_col_profile(_vp(m), m.shape[0], m.shape[1], max(m.shape[0], 1),
                                               _lib.STAT[avgfun], 1 if scale == "log2" else 0,
                                               _lib.MEM_HOST, _vp(center), _vp(spread)))
    return center, spread


def calcPlotProfiles(input, opts, sdim=2, rc=None):
    """plot.R:949-990 without the smoothing branch: one dict(profile, upper, lower) per sample.
    smooth = TRUE (smooth.spline + its confidence band) is plotting-side statistics and not part
    of this library."""
    pp = opts["plotParams"]
    if pp.get("smooth"):
        raise NotImplementedError("plotParams$smooth: smooth.spline is outside the accelerated path")
    if sdim != 2:
        raise NotImplementedError("only column profiles (sdim = 2) are used by recoup")
    out = []
    for x in input:
        center, spread = colProfile(x["profile"], pp.get("sumStat", "mean"), pp.get("signalScale", "natural"))
        out.append({"profile": center, "upper": center + spread, "lower": center - spread})
    return out


def groupColProfile(mat, codes, n_groups, avgfun="mean", scale="natural"):
    """colProfile of every group of rows (rcp_matrix_group_col_profile): row i belongs to group
    codes[i], 1-based as R stores a factor; a code <= 0 excludes the row; codes None puts every
    row in group 1.  Returns (center, spread), each n_groups x n_cols; a group without rows is NaN."""
    if avgfun not in ("mean", "median"):
        raise ValueError("sumStat must be mean or median")
    m = _f(mat)
    c = None
    if codes is not None:
        c = np.ascontiguousarray(codes, dtype=np.int32)
        if c.shape != (m.shape[0],):
            raise ValueError("%d codes for %d rows" % (c.size, m.shape[0]))
    g = int(n_groups)
    _lib.ensure_init()
    center = np.empty((max(g, 0), m.shape[1]), dtype=np.float64, order="F")
    spread = np.empty((max(g, 0), m.shape[1]), dtype=np.float64, order="F")
    _lib.check(_lib.lib.rcp_matrix_group_col_profile(_vp(m), m.shape[0], m.shape[1], max(m.shape[0], 1),
                                                     None if c is None else _vp(c), g, _lib.STAT[avgfun],
                                                     1 if scale == "log2" else 0, _lib.MEM_HOST, _vp(center),
                                                     _vp(spread)))
    return center, spread


def _design_levels(design, n_rows):
    """The levels of a design (dict of equal-length label columns): the label, or the tuple of
    labels across columns, of every combination that occurs, ordered as factor() orders each
    column (sorted labels), first column slowest; a row with a None label is in no level.
    Returns (levels, codes): codes[i] is the 1-based level of row i, 0 when excluded."""
    if not design:
        raise ValueError("calcDesignPlotProfiles needs a design with at least one column")
    cols = [np.asarray(v, dtype=object) for v in design.values()]
    for name, v in zip(design, cols):
        if v.ndim != 1 or v.shape[0] != n_rows:
            raise ValueError("design column %s has %d rows, the profiles %d" % (name, v.size, n_rows))
    keep = np.ones(n_rows, dtype=bool)
    for v in cols:
        keep &= np.array([lab is not None for lab in v.tolist()], dtype=bool)
    ranks = []
    for v in cols:
        labels = sorted(set(v[keep].tolist()))
        pos = {lab: i for i, lab in enumerate(labels)}
        ranks.append(np.array([pos[lab] if k else -1 for lab, k in zip(v.tolist(), keep)], dtype=np.int64))
    combo = {}
    for i in np.flatnonzero(keep):
        key = tuple(int(r[i]) for r in ranks)
        if key not in combo:
            combo[key] = tuple(v[i] for v in cols)
    order = sorted(combo)
    code_of = {key: j + 1 for j, key in enumerate(order)}
    codes = np.zeros(n_rows, dtype=np.int32)
    for i in np.flatnonzero(keep):
        codes[i] = code_of[tuple(int(r[i]) for r in ranks)]
    levels = [combo[key][0] if len(cols) == 1 else combo[key] for key in order]
    return levels, codes


def _group_profiles(mats, codes, n_groups, avgfun, log2):
    """(center, spread) of rcp_matrix_group_col_profile for every matrix, each n_groups x n_cols;
    the codes are uploaded once, every matrix is staged and reduced on the device."""
    import torch
    _lib.ensure_init()
    dev = torch.device("cuda", _lib._initialised_device)
    d_codes = torch.from_numpy(np.ascontiguousarray(codes, dtype=np.int32)).to(dev)
    out = []
    for m in mats:
        dm = torch.from_numpy(np.ascontiguousarray(m.T)).to(dev)        # m^T row-major = m column-major
        center = torch.empty((m.shape[1], n_groups), dtype=torch.float64, device=dev)
        spread = torch.empty_like(center)
        torch.cuda.synchronize(dev)
        _lib.check(_lib.lib.rcp_matrix_group_col_profile(
            C.c_void_p(dm.data_ptr()), m.shape[0], m.shape[1], max(m.shape[0], 1), C.c_void_p(d_codes.data_ptr()),
            n_groups, _lib.STAT[avgfun], log2, _lib.MEM_DEVICE, C.c_void_p(center.data_ptr()),
            C.c_void_p(spread.data_ptr())))
        _lib.check(_lib.lib.rcp_sync())
        out.append((center.cpu().numpy().T, spread.cpu().numpy().T))
    return out


def calcDesignPlotProfiles(input, design, opts):
    """The curves of a design-split profile plot (calcDesignPlotProfiles, parity unpinned): for
    every level of `design` (see _design_levels; kmeansDesign's result can be passed as is) and
    every sample, calcPlotProfiles over that level's rows.  Returns one (level, rows (1-based
    int32), [dict(profile, upper, lower) per sample]) per level.  The level codes go to the
    device once and serve every sample."""
    pp = opts["plotParams"]
    if pp.get("smooth"):
        raise NotImplementedError("plotParams$smooth: smooth.spline is outside the accelerated path")
    avgfun = pp.get("sumStat", "mean")
    if avgfun not in ("mean", "median"):
        raise ValueError("sumStat must be mean or median")
    log2 = 1 if pp.get("signalScale", "natural") == "log2" else 0
    n_rows = np.asarray(input[0]["profile"]).shape[0] if input else 0
    levels, codes = _design_levels(design, n_rows)
    G = len(levels)
    rows = [(np.flatnonzero(codes == j + 1) + 1).astype(np.int32) for j in range(G)]
    curves = [[] for _ in range(G)]
    if G and input:
        mats = [_f(x["profile"]) for x in input]
        for m in mats:
            if m.shape[0] != n_rows:
                raise ValueError("every sample's profile must have %d rows" % n_rows)
        for cen, spr in _group_profiles(mats, codes, G, avgfun, log2):
            for j in range(G):
                curves[j].append({"profile": cen[j].copy(), "upper": cen[j] + spr[j], "lower": cen[j] - spr[j]})
    return [(levels[j], rows[j], curves[j]) for j in range(G)]


def rowStat(mat, what):
    """apply(x, 1, sum | max | mean)"""
    m = _f(mat)
    _lib.ensure_init()
    out = np.empty(m.shape[0], dtype=np.float64)
    _lib.check(_lib.lib.rcp_matrix_row_stat(_vp(m), m.shape[0], m.shape[1], max(m.shape[0], 1),
                                            _ROW[what], _lib.MEM_HOST, _vp(out)))
    return out


def sortIndex(v, decreasing=False):
    """sort(v, decreasing, index.return=TRUE): dict(x = sorted values, ix = 1-based positions)"""
    v = np.ascontiguousarray(v, dtype=np.float64)
    _lib.ensure_init()
    ix = np.empty(v.shape[0], dtype=np.int32)
    n_out = C.c_int64(0)
    _lib.check(_lib.lib.rcp_order(_vp(v), v.shape[0], 1 if decreasing else 0, _lib.MEM_HOST, _vp(ix),
                                  C.byref(n_out)))
    ix = ix[:n_out.value]
    return {"x": v[ix - 1], "ix": ix}


def orderProfiles(input, opts, rc=None):
    """plot.R:1035-1150.  orderBy$what = "sum" | "max" | "avg" followed by the 1-based number of
    the reference sample, or by "a" for all samples together; anything else keeps the input
    order; orderBy$custom overrides everything."""
    ob = opts["orderBy"]
    dec = ob.get("order") == "descending"
    if ob.get("custom") is not None:
        return sortIndex(ob["custom"], dec)
    what = ob.get("what", "none")
    m = re.match(r"^(sum|max|avg)", what)
    if not m:
        n = np.asarray(input[0]["profile"]).shape[0]
        return {"ix": np.arange(1, n + 1, dtype=np.int32)}
    kind = m.group(1)
    ref = 1
    last = what[-1]
    if last == "a":
        ref = 0
    elif last.isdigit():
        ref = int(last)
    if ref == 0:
        per = np.stack([rowStat(x["profile"], kind) for x in input], axis=1)
        val = rowStat(per, kind)
    else:
        val = rowStat(input[ref - 1]["profile"], kind)
    return sortIndex(val, dec)


def matrixQuantile(mat, probs):
    """quantile(x, probs), type 7, over every cell"""
    m = _f(mat)
    _lib.ensure_init()
    p = np.ascontiguousarray(np.atleast_1d(probs), dtype=np.float64)
    out = np.empty(p.shape[0], dtype=np.float64)
    _lib.check(_lib.lib.rcp_matrix_quantile(_vp(m), m.shape[0], m.shape[1], max(m.shape[0], 1), _vp(p),
                                            p.shape[0], _lib.MEM_HOST, _vp(out)))
    return out


_QS = (0.95, 0.96, 0.97, 0.98, 0.99, 0.995, 0.999)


def heatmapScale(input, heatmapScale="common", heatmapFactor=1.0):
    """Upper colour limit of every sample's heat map (plot.R:513-545): "each" walks up the
    quantile ladder until it is non-zero; "common" takes the largest 95 % quantile."""
    if heatmapScale == "each":
        out = []
        for x in input:
            qs = matrixQuantile(x["profile"], _QS)
            nz = [q for q in qs if q != 0]
            out.append(heatmapFactor * (nz[0] if nz else 0.0))
        return out
    sup = max(float(matrixQuantile(x["profile"], [0.95])[0]) for x in input)
    return [heatmapFactor * sup] * len(input)


_KM_ALGORITHMS = ("Hartigan-Wong", "Lloyd", "Forgy", "MacQueen")
_KM_CODE = {"Hartigan-Wong": 1, "Lloyd": 2, "Forgy": 2, "MacQueen": 3}


class NamedVector(np.ndarray):
    """A vector carrying R's names attribute (`names`, None when unnamed)."""

    def __new__(cls, array, names=None):
        obj = np.asarray(array).view(cls)
        obj.names = names
        return obj

    def __array_finalize__(self, obj):
        if obj is not None:
            self.names = getattr(obj, "names", None)


def _match_algorithm(algorithm):
    """match.arg(algorithm): exact name or unique prefix; "Forgy" is "Lloyd"."""
    if isinstance(algorithm, (list, tuple)):
        algorithm = algorithm[0]
    if algorithm in _KM_ALGORITHMS:
        return algorithm
    hits = [a for a in _KM_ALGORITHMS if algorithm and a.startswith(algorithm)]
    if len(hits) != 1:
        raise ValueError("'arg' should be one of %s" % ", ".join('"%s"' % a for a in _KM_ALGORITHMS))
    return hits[0]


def kmeans(x, centers, iter_max=10, nstart=1, algorithm="Hartigan-Wong", seed=42, sample_kind="Rejection"):
    """`set.seed(seed); kmeans(x, centers, iter.max, nstart, algorithm)` on the device
    (rcp_kmeans).  `centers` is the number of clusters.  Returns dict(cluster (1-based, named by
    x.rownames for a ProfileMatrix), centers (k x p), totss, withinss, tot_withinss, betweenss,
    size, iter, ifault) and raises R's warnings."""
    if isinstance(centers, (bool, np.bool_)) or not isinstance(centers, (int, np.integer)):
        raise TypeError("centers must be the number of clusters")
    algorithm = _match_algorithm(algorithm)
    m = _f(x)
    n, p = m.shape
    k = int(centers)
    _lib.ensure_init()
    cluster = np.empty(n, dtype=np.int32)
    cen = np.empty((max(k, 0), p), dtype=np.float64, order="F")
    wss = np.empty(max(k, 0), dtype=np.float64)
    size = np.empty(max(k, 0), dtype=np.int32)
    totss = C.c_double(0.0)
    it, ifault, warn = C.c_int(0), C.c_int(0), C.c_int(0)
    _lib.check(_lib.lib.rcp_kmeans(_vp(m), n, p, max(n, 1), k, int(nstart), int(iter_max), _KM_CODE[algorithm],
                                   int(seed), _lib.SAMPLE_KIND[sample_kind], _lib.MEM_HOST, _vp(cluster), _vp(cen),
                                   _vp(wss), _vp(size), C.byref(totss), C.byref(it), C.byref(ifault),
                                   C.byref(warn)))
    w = warn.value
    if w & 1:
        warnings.warn("did not converge in %d iteration%s" % (iter_max, "" if iter_max == 1 else "s"),
                      stacklevel=2)
    if w & 4:
        warnings.warn("Quick-TRANSfer stage steps exceeded maximum (= %d)" % min(2147483647, 50 * n),
                      stacklevel=2)
    if w & 2:
        warnings.warn("empty cluster: try a better set of initial centers", stacklevel=2)
    tot_w = float(np.sum(wss.astype(np.longdouble)))
    return {"cluster": NamedVector(cluster, getattr(x, "rownames", None)), "centers": cen,
            "totss": totss.value, "withinss": wss, "tot_withinss": tot_w, "betweenss": totss.value - tot_w,
            "size": size, "iter": it.value, "ifault": ifault.value}


_KM_DEFAULTS = {"k": 0, "nstart": 20, "algorithm": "Hartigan-Wong", "iterMax": 20, "reference": None, "seed": 42}


def kmeansDesign(input, design=None, kmParams=None):
    """util.R:140-197 (parity unpinned): split the heat map into k-means clusters.  kmParams =
    dict(k, nstart, algorithm, iterMax, reference, seed) over the defaults above; k == 0 returns
    `design` unchanged.  The matrix is the profile of the sample whose `id` is `reference`, else
    the cbind of every sample's profile in sample order (an unknown reference warns and uses all
    samples).  Returns the design -- a dict of equal-length columns, created when None -- with a
    `Cluster` column of "Cluster <n>" labels, one per row in row order."""
    kp = dict(_KM_DEFAULTS)
    kp.update(kmParams or {})
    if int(kp["k"]) == 0:
        return design
    ref = kp.get("reference")
    mats = None
    if ref is not None:
        ids = [s.get("id") for s in input]
        if ref in ids:
            mats = [input[ids.index(ref)]["profile"]]
        else:
            warnings.warn("reference %s not found in the input sample ids; using all samples for k-means "
                          "clustering" % ref, stacklevel=2)
    if mats is None:
        mats = [s["profile"] for s in input]
    x = np.asfortranarray(np.hstack([np.asarray(mm, dtype=np.float64) for mm in mats]))
    names = getattr(mats[0], "rownames", None)
    if names is not None:
        from .profile import ProfileMatrix
        x = ProfileMatrix(x, rownames=names)
    km = kmeans(x, int(kp["k"]), iter_max=int(kp["iterMax"]), nstart=int(kp["nstart"]),
                algorithm=kp["algorithm"], seed=int(kp["seed"]))
    labels = np.array(["Cluster %d" % c for c in np.asarray(km["cluster"])], dtype=object)
    out = {} if design is None else dict(design)
    for col, v in out.items():
        if len(v) != labels.shape[0]:
            raise ValueError("design column %s has %d rows, the profiles %d" % (col, len(v), labels.shape[0]))
    out["Cluster"] = labels
    return out


_HC_METHODS = ("ward.D", "single", "complete", "average", "mcquitty", "median", "centroid", "ward.D2")


def hclust(x, method="complete"):
    """`hclust(dist(x), method)` on the device (rcp_hclust): Euclidean distances of the rows, then
    the merges of hclust.f, bit for bit as R computes them.  Only method = "complete" (hclust's
    default, and ComplexHeatmap's) is implemented.  Returns dict(merge ((n-1) x 2, R's signs),
    height, order (1-based), labels (x.rownames for a ProfileMatrix, else None), method,
    dist_method)."""
    if method == "ward":
        method = "ward.D"
    hits = [mm for mm in _HC_METHODS if mm == method] or [mm for mm in _HC_METHODS if method and
                                                          mm.startswith(method)]
    if not hits:
        raise ValueError("invalid clustering method %s" % method)
    if len(hits) > 1:
        raise ValueError("ambiguous clustering method %s" % method)
    m = _f(x)
    n, p = m.shape
    _lib.ensure_init()
    merge = np.empty(2 * max(n - 1, 1), dtype=np.int32)
    height = np.empty(max(n - 1, 1), dtype=np.float64)
    order = np.empty(max(n, 1), dtype=np.int32)
    _lib.check(_lib.lib.rcp_hclust(_vp(m), n, p, max(n, 1), _HC_METHODS.index(hits[0]) + 1, _lib.MEM_HOST,
                                   _vp(merge), _vp(height), _vp(order)))
    return {"merge": merge.reshape((n - 1, 2), order="F"), "height": height, "order": order,
            "labels": getattr(x, "rownames", None), "method": hits[0], "dist_method": "euclidean"}


def heatmapClusters(input, opts, split=None):
    """The row dendrograms of recoup's heat maps (cluster_rows) for opts["orderBy"]["what"] =
    "hc<n>" (the profile of sample n, 1-based) or "hca" (the cbind of every sample's profile in
    sample order, as kmeansDesign builds it); any other `what` returns None, and orderBy$order
    does not apply to a dendrogram.  Without `split` the result is hclust() of that matrix.  With
    `split` (one label per row, e.g. a design column or kmeansDesign's Cluster) every level's rows
    are clustered on their own, as ComplexHeatmap does with row_split: a list of (level, rows
    (1-based), hclust) per level in factor() order (sorted labels); a one-row level gets None."""
    what = opts["orderBy"].get("what", "none")
    m = re.match(r"^hc(\d+|a)$", what or "")
    if not m:
        return None
    if m.group(1) == "a":
        mats = [s["profile"] for s in input]
    else:
        ref = int(m.group(1))
        if not 1 <= ref <= len(input):
            raise ValueError("orderBy$what = %s: there are %d samples" % (what, len(input)))
        mats = [input[ref - 1]["profile"]]
    names = getattr(mats[0], "rownames", None)
    x = np.asfortranarray(np.hstack([np.asarray(mm, dtype=np.float64) for mm in mats]))
    if split is None:
        if names is not None:
            from .profile import ProfileMatrix
            x = ProfileMatrix(x, rownames=names)
        return hclust(x)
    lab = np.asarray(split, dtype=object)
    if lab.shape[0] != x.shape[0]:
        raise ValueError("split has %d labels, the profiles %d rows" % (lab.shape[0], x.shape[0]))
    out = []
    for level in sorted(set(lab.tolist())):
        rows = np.flatnonzero(lab == level)
        hc = None
        if rows.shape[0] >= 2:
            sub = np.asfortranarray(x[rows])
            if names is not None:
                from .profile import ProfileMatrix
                sub = ProfileMatrix(sub, rownames=[names[r] for r in rows])
            hc = hclust(sub)
        out.append((level, (rows + 1).astype(np.int32), hc))
    return out
