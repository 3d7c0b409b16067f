"""hclust(dist(x), "complete") for the heat-map rows of orderBy = "hc<n>" / "hca": the C
restatement of R_euclidean / hclust.f / HCASS2 (oracle/hclust_oracle.c) against a brute-force
definition and a hand-solved answer on the CPU, the host logic of heatmapClusters, and rcp_hclust
against the restatement, bit for bit, under `-m gpu` on a B200."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from oracle import hclust_oracle as H


# ---------------------------------------------------------------- independent definitions -----
def py_dist(x):
    """R_euclidean in a Python loop: columns in order, then sqrt; full n x n."""
    n, p = x.shape
    d = np.zeros((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            s = 0.0
            for c in range(p):
                t = float(x[i, c]) - float(x[j, c])
                s += t * t
            d[i, j] = d[j, i] = math.sqrt(s)
    return d


def condensed(d):
    n = d.shape[0]
    return np.array([d[i, j] for j in range(n) for i in range(j + 1, n)])


def brute(d):
    """Complete linkage by its definition: merge the alive pair with the smallest distance, ties by
    the smaller i, then the smaller j, into i.  1-based ia / ib and the heights."""
    n = d.shape[0]
    d = d.copy()
    alive = list(range(n))
    ia, ib, crit = [], [], []
    while len(alive) > 1:
        best = min((d[i, j], i, j) for a, i in enumerate(alive) for j in alive[a + 1:])
        h, i, j = best
        ia.append(i + 1)
        ib.append(j + 1)
        crit.append(h)
        alive.remove(j)
        for k in alive:
            if k != i:
                d[i, k] = d[k, i] = max(d[i, k], d[j, k])
    return ia, ib, crit


def tie_heavy(rng, trial):
    n = int(rng.integers(2, 61))
    p = int(rng.integers(1, 5))
    kind = trial % 6
    if kind == 0:                                    # small integers
        x = rng.integers(0, 3, size=(n, p)).astype(float)
    elif kind == 1:                                  # duplicate rows
        base = rng.integers(0, 4, size=(max(1, n // 4), p)).astype(float)
        x = base[rng.integers(0, base.shape[0], size=n)]
    elif kind == 2:                                  # zero rows among gaussians
        x = rng.normal(size=(n, p))
        x[rng.random(n) < 0.4] = 0.0
    elif kind == 3:                                  # a single column
        x = rng.integers(0, 5, size=(n, 1)).astype(float)
    elif kind == 4:                                  # all rows equal
        x = np.tile(rng.normal(size=(1, p)), (n, 1))
    else:
        x = np.round(rng.normal(size=(n, p)), 1)
    return np.asfortranarray(x)


def check_well_formed(merge, height, order, n):
    """R's conventions: singletons negative, clusters their positive step, a singleton first in a
    mixed row, two clusters ascending; every step used once; order a permutation in which every
    cluster's leaves are contiguous; heights non-decreasing (complete linkage is monotone)."""
    assert merge.shape == (n - 1, 2)
    used = set()
    leaves = {}
    for s, (a, b) in enumerate(merge.tolist(), start=1):
        if a > 0 and b > 0:
            assert a < b
        assert not (a > 0 and b < 0)
        for v in (a, b):
            assert v != 0 and v not in used
            assert v < s
            used.add(v)
        leaves[s] = (leaves[a] if a > 0 else [-a]) + (leaves[b] if b > 0 else [-b])
    assert sorted(-v for v in used if v < 0) == list(range(1, n + 1))
    assert sorted(order.tolist()) == list(range(1, n + 1))
    pos = {v: i for i, v in enumerate(order.tolist())}
    for s, lv in leaves.items():
        ps = sorted(pos[v] for v in lv)
        assert ps[-1] - ps[0] == len(ps) - 1, s
    assert np.all(np.diff(height) >= 0)


def closed_form(n):
    """x = 0..n-1 in one column, n = 2^m: round r merges neighbouring clusters at height 2^r - 1."""
    merge, height = [], []
    merge += [(-(2 * a + 1), -(2 * a + 2)) for a in range(n // 2)]
    height += [1.0] * (n // 2)
    base, m, r = 0, n // 2, 2
    while m > 1:
        merge += [(base + 2 * a + 1, base + 2 * a + 2) for a in range(m // 2)]
        height += [2.0 ** r - 1] * (m // 2)
        base += m
        m //= 2
        r += 1
    return np.array(merge, dtype=np.int32), np.array(height), np.arange(1, n + 1, dtype=np.int32)


# ---------------------------------------------------------------- oracle on the CPU -----------
def test_oracle_dist_equals_python_loop():
    rng = np.random.default_rng(3)
    for n, p in ((2, 1), (7, 3), (40, 17)):
        x = np.asfortranarray(rng.normal(size=(n, p)) * 10.0 ** rng.integers(-3, 4, size=(n, p)))
        got = H.dist(x)
        want = condensed(py_dist(x))
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


def test_oracle_equals_brute_force_on_tie_heavy_cases():
    rng = np.random.default_rng(11)
    for trial in range(300):
        x = tie_heavy(rng, trial)
        n = x.shape[0]
        ia, ib, crit = H.hclust_dist(H.dist(x), n)
        bia, bib, bcrit = brute(py_dist(x))
        assert ia.tolist() == bia and ib.tolist() == bib, trial
        assert np.array_equal(crit, np.array(bcrit)), trial
        merge, order = H.hcass2(n, ia, ib)
        check_well_formed(merge, crit, order, n)


def test_closed_form_known_answer():
    for n in (2, 4, 64, 256):
        got = H.hclust(np.arange(n, dtype=np.float64)[:, None])
        merge, height, order = closed_form(n)
        np.testing.assert_array_equal(got["merge"], merge)
        np.testing.assert_array_equal(got["height"], height)
        np.testing.assert_array_equal(got["order"], order)
    merge, _, _ = closed_form(64)
    assert merge[0].tolist() == [-1, -2] and merge[1].tolist() == [-3, -4]
    assert merge[32].tolist() == [1, 2] and merge[-1].tolist() == [61, 62]


def test_hcass2_small_known_answer():
    # x = (0, 10, 11, 30): 2 and 3 join at 1, then 1 with {2,3} at 11, then 4 at 30
    got = H.hclust(np.array([[0.0], [10.0], [11.0], [30.0]]))
    assert got["merge"].tolist() == [[-2, -3], [-1, 1], [-4, 2]]
    assert got["height"].tolist() == [1.0, 11.0, 30.0]
    assert got["order"].tolist() == [4, 1, 2, 3]


def test_oracle_refuses_bad_input():
    with pytest.raises(H.HclustError, match="must have n >= 2 objects"):
        H.hclust(np.zeros((1, 3)))
    with pytest.raises(H.HclustError, match="NA/NaN/Inf"):
        H.hclust(np.array([[0.0], [np.nan], [1.0]]))
    with pytest.raises(H.HclustError, match="1e300"):
        H.hclust(np.array([[1e299], [-1e299]]))


# ---------------------------------------------------------------- heatmapClusters (host) ------
@pytest.fixture
def oracle_hclust(monkeypatch):
    """heatmapClusters with the restatement standing in for the device call; records the matrices."""
    from recoup_b200 import consumers
    seen = []

    def fake(x, method="complete"):
        seen.append(np.array(x))
        out = H.hclust(np.asarray(x))
        out["labels"] = getattr(x, "rownames", None)
        return out
    monkeypatch.setattr(consumers, "hclust", fake)
    return seen


def _input():
    from recoup_b200 import ProfileMatrix
    rng = np.random.default_rng(2)
    names = ["g%d" % i for i in range(9)]
    return [dict(id="A", profile=ProfileMatrix(rng.integers(0, 3, size=(9, 4)).astype(float), rownames=names)),
            dict(id="B", profile=ProfileMatrix(rng.integers(0, 3, size=(9, 5)).astype(float), rownames=names))]


def test_heatmap_clusters_choice_of_matrix(oracle_hclust):
    from recoup_b200 import heatmapClusters
    inp = _input()
    got = heatmapClusters(inp, dict(orderBy=dict(what="hc2", order="descending")))
    assert np.array_equal(oracle_hclust[-1], np.asarray(inp[1]["profile"]))
    assert got["labels"] == ["g%d" % i for i in range(9)]
    heatmapClusters(inp, dict(orderBy=dict(what="hc1")))
    assert np.array_equal(oracle_hclust[-1], np.asarray(inp[0]["profile"]))
    got = heatmapClusters(inp, dict(orderBy=dict(what="hca")))
    both = np.hstack([np.asarray(s["profile"]) for s in inp])
    assert np.array_equal(oracle_hclust[-1], both)
    np.testing.assert_array_equal(got["order"], H.hclust(both)["order"])
    for what in ("none", "sum1", "hc", "hcb", "max", "hc1x"):
        assert heatmapClusters(inp, dict(orderBy=dict(what=what))) is None
    with pytest.raises(ValueError, match="there are 2 samples"):
        heatmapClusters(inp, dict(orderBy=dict(what="hc3")))


def test_heatmap_clusters_split_levels(oracle_hclust):
    from recoup_b200 import heatmapClusters
    inp = _input()
    split = ["b", "a", "b", "c", "a", "b", "a", "b", "a"]          # "c" has one row
    got = heatmapClusters(inp, dict(orderBy=dict(what="hca")), split=split)
    assert [lv for lv, _, _ in got] == ["a", "b", "c"]
    both = np.hstack([np.asarray(s["profile"]) for s in inp])
    for level, rows, hc in got:
        want_rows = [i + 1 for i, s in enumerate(split) if s == level]
        assert rows.tolist() == want_rows
        if len(want_rows) == 1:
            assert hc is None
            continue
        want = H.hclust(both[rows - 1])
        np.testing.assert_array_equal(hc["merge"], want["merge"])
        np.testing.assert_array_equal(hc["order"], want["order"])
        assert hc["labels"] == ["g%d" % (r - 1) for r in rows]
    with pytest.raises(ValueError, match="split has 3 labels"):
        heatmapClusters(inp, dict(orderBy=dict(what="hc1")), split=["a", "b", "c"])


# ---------------------------------------------------------------- on the device --------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import recoup_b200 as rb
    rb.init(0)
    return rb


def blobs(n, p, k, seed, zero_frac=0.0):
    rng = np.random.default_rng(seed)
    cen = rng.normal(size=(k, p)) * 3.0
    x = cen[rng.integers(0, k, size=n)] + rng.normal(size=(n, p))
    x[rng.random(n) < zero_frac] = 0.0
    return np.asfortranarray(x)


def c1_profiles():
    from tests.test_kmeans import fixture_c1_profiles
    return fixture_c1_profiles()


INPUTS = {
    "blobs": lambda: blobs(500, 6, 5, 1),
    "c1": c1_profiles,
    "ties012": lambda: np.asfortranarray(np.random.default_rng(4).integers(0, 3, size=(900, 5)).astype(float)),
    "identical": lambda: np.asfortranarray(np.tile(np.random.default_rng(5).normal(size=(1, 4)), (300, 1))),
    "n2": lambda: blobs(2, 3, 1, 6),
    "n3": lambda: np.array([[0.0, 1.0], [0.0, 1.0], [2.0, 0.0]]),
    "n1000_p200": lambda: blobs(1000, 200, 6, 7, zero_frac=0.1),
    "p1": lambda: np.asfortranarray(np.round(np.random.default_rng(8).normal(size=(700, 1)), 2)),
    "p3000": lambda: blobs(150, 3000, 3, 9, zero_frac=0.1),
    "n20000_p200": lambda: blobs(20_000, 200, 8, 10, zero_frac=0.1),
}


def assert_same(got, want):
    np.testing.assert_array_equal(got["merge"], want["merge"])
    np.testing.assert_array_equal(got["order"], want["order"])
    assert np.array_equal(np.asarray(got["height"]).view(np.uint64), np.asarray(want["height"]).view(np.uint64))


@gpu
@pytest.mark.parametrize("name", list(INPUTS))
def test_device_equals_oracle(rb, name):
    x = INPUTS[name]()
    got = rb.hclust(x)
    want = H.hclust(x)
    assert_same(got, want)
    assert got["method"] == "complete" and got["dist_method"] == "euclidean" and got["labels"] is None


def _call(x_ptr, n, p, ld, mem, merge, height, order, method=3):
    from recoup_b200 import _lib
    return _lib.lib.rcp_hclust(x_ptr, n, p, ld, method, mem, merge, height, order)


@gpu
def test_row_block_of_taller_matrix(rb):
    from recoup_b200 import _lib
    tall = blobs(1300, 40, 4, 12, zero_frac=0.1)
    n, p = 1000, 40
    merge = np.zeros(2 * (n - 1), np.int32)
    height = np.zeros(n - 1)
    order = np.zeros(n, np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    _lib.check(_call(vp(tall), n, p, tall.shape[0], _lib.MEM_HOST, vp(merge), vp(height), vp(order)))
    want = H.hclust(tall[:n])
    assert_same(dict(merge=merge.reshape((n - 1, 2), order="F"), height=height, order=order), want)


@gpu
def test_host_and_device_memory_agree(rb):
    import torch
    from recoup_b200 import _lib
    x = blobs(2000, 30, 5, 13, zero_frac=0.1)
    want = rb.hclust(x)
    n, p = x.shape
    xd = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    merge = torch.empty(2 * (n - 1), dtype=torch.int32, device="cuda")
    height = torch.empty(n - 1, dtype=torch.float64, device="cuda")
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    _lib.check(_call(C.c_void_p(xd.data_ptr()), n, p, n, _lib.MEM_DEVICE, C.c_void_p(merge.data_ptr()),
                     C.c_void_p(height.data_ptr()), C.c_void_p(order.data_ptr())))
    _lib.check(_lib.lib.rcp_sync())
    assert_same(dict(merge=merge.cpu().numpy().reshape((n - 1, 2), order="F"), height=height.cpu().numpy(),
                     order=order.cpu().numpy()), want)


@gpu
def test_closed_form_at_r_limit(rb):
    n = 65536
    got = rb.hclust(np.arange(n, dtype=np.float64)[:, None])
    merge, height, order = closed_form(n)
    np.testing.assert_array_equal(got["merge"], merge)
    np.testing.assert_array_equal(got["height"], height)
    np.testing.assert_array_equal(got["order"], order)


def pool_used():
    """cudaMemPoolAttrUsedMemCurrent of device 0's default pool (driver API)."""
    cu = C.CDLL("libcuda.so.1")
    dev, pool, val = C.c_int(0), C.c_void_p(0), C.c_uint64(0)
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    assert cu.cuMemPoolGetAttribute(pool, 7, C.byref(val)) == 0      # CU_MEMPOOL_ATTR_USED_MEM_CURRENT
    return val.value


@gpu
def test_errors_leave_no_memory_behind(rb):
    from recoup_b200 import _lib
    vp = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    buf = np.zeros(4 * 65537, np.int32)
    hb = np.zeros(65537)
    x = np.zeros(65537)

    def code(xx, n, p, ld, method=3, mem=_lib.MEM_HOST):
        _lib.check(_lib.lib.rcp_sync())
        before = pool_used()
        rc = _call(vp(xx), n, p, ld, mem, vp(buf), vp(hb), vp(buf), method)
        msg = _lib.lib.rcp_last_error().decode()
        _lib.check(_lib.lib.rcp_sync())
        assert pool_used() == before, (n, p, msg)
        return rc, msg

    assert code(x, 1, 1, 1) == (_lib.RCP_ERR_ARG, "must have n >= 2 objects to cluster")
    assert code(x, 0, 1, 1)[0] == _lib.RCP_ERR_ARG
    assert code(x, 65537, 1, 65537) == (_lib.RCP_ERR_ARG, "size cannot be NA nor exceed 65536")
    assert code(x, 10, 0, 10)[0] == _lib.RCP_ERR_ARG
    assert code(x, 10, 2, 9)[0] == _lib.RCP_ERR_ARG
    assert code(x, 10, 1, 10, mem=7)[0] == _lib.RCP_ERR_ARG
    for method in (1, 2, 4, 5, 6, 7, 8, 0):
        assert code(x, 10, 1, 10, method=method)[0] == _lib.RCP_ERR_UNSUPPORTED
    bad = np.zeros(20)
    for v in (np.nan, np.inf, -np.inf):
        bad[13] = v
        rc, msg = code(bad, 10, 2, 10)
        assert rc == _lib.RCP_ERR_DATA and "NA/NaN/Inf" in msg
    big = np.array([1e299, 0.0, -1e299])
    rc, msg = code(big, 3, 1, 3)
    assert rc == _lib.RCP_ERR_DATA and "1e300" in msg
    with pytest.raises(ValueError, match="invalid clustering method"):
        rb.hclust(np.zeros((3, 1)), "nosuch")
    with pytest.raises(ValueError, match="ambiguous clustering method"):
        rb.hclust(np.zeros((3, 1)), "ward.")
    with pytest.raises(rb.RecoupError) as ei:
        rb.hclust(np.zeros((3, 1)), "average")
    assert ei.value.code == _lib.RCP_ERR_UNSUPPORTED


@gpu
def test_heatmap_clusters_on_device_profiles(rb):
    from tests.helpers import fixture_genes, fixture_reads
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "recoup_test_data.npz"))
    _, g_genes = fixture_genes(z)
    inp = []
    for s, name in enumerate(("WT", "KO")):
        _, g_reads = fixture_reads(z, s)
        inp.append(dict(id=name, name=name, ranges=g_reads))
    rb.coverageRef(inp, g_genes, "tss", (2000, 2000))
    rb.profileMatrix(inp, (2000, 2000), dict(flankBinSize=0, regionBinSize=100, sumStat="mean",
                                             interpolation="auto"))
    opts = dict(orderBy=dict(what="hc1"))
    one = rb.heatmapClusters(inp, opts)
    assert_same(one, H.hclust(np.asarray(inp[0]["profile"])))
    assert one["labels"] == inp[0]["profile"].rownames
    both = np.hstack([np.asarray(s["profile"]) for s in inp])
    assert_same(rb.heatmapClusters(inp, dict(orderBy=dict(what="hca"))), H.hclust(both))
    n = both.shape[0]
    design = np.array(["up" if i % 3 else "down" for i in range(n)], dtype=object)
    design[5] = "single"
    got = rb.heatmapClusters(inp, opts, split=design)
    assert [lv for lv, _, _ in got] == ["down", "single", "up"]
    for level, rows, hc in got:
        assert rows.tolist() == [i + 1 for i in range(n) if design[i] == level]
        if rows.shape[0] == 1:
            assert hc is None
        else:
            assert_same(hc, H.hclust(np.asarray(inp[0]["profile"])[rows - 1]))
