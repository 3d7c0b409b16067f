"""kmeans / kmeansDesign (util.R:140-197): the draws of stats::kmeans, unique(x), the C restatement
of its three algorithms (oracle/kmeans_oracle.c) and the host logic of kmeansDesign on the CPU;
rcp_kmeans against that restatement, bit for bit, under `-m gpu` on a B200."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

from oracle import kmeans_oracle as K
from oracle.r_rng import RRandom

ALGS = ["Hartigan-Wong", "Lloyd", "MacQueen"]


# ---------------------------------------------------------------- draws ----------------------
def test_sample_int_known_answer():
    # set.seed(42); sample.int(10, 3) is the prefix of the known sample(1:10) = 1 5 10 8 2 ...
    assert RRandom(42).sample_int(10, 3) == [1, 5, 10]
    from recoup_b200 import _lib
    out = np.zeros(3, dtype=np.int32)
    n, k = np.array([10], np.int64), np.array([3], np.int64)
    _lib.check(_lib.lib.rcp_r_sample_int(42, 0, 1, n.ctypes.data_as(C.POINTER(C.c_int64)),
                                         k.ctypes.data_as(C.POINTER(C.c_int64)), out.ctypes.data_as(C.c_void_p)))
    assert out.tolist() == [1, 5, 10]


@pytest.mark.parametrize("kind", ["Rejection", "Rounding"])
def test_sample_int_stream_of_starts(kind):
    """nstart draws of sample.int(mm, k) come from ONE stream, unsorted, in draw order."""
    from recoup_b200 import _lib
    n = np.array([97, 97, 97, 20_000_001, 5], np.int64)
    k = np.array([5, 5, 5, 4, 5], np.int64)
    out = np.zeros(int(k.sum()), dtype=np.int32)
    _lib.check(_lib.lib.rcp_r_sample_int(7, _lib.SAMPLE_KIND[kind], n.shape[0],
                                         n.ctypes.data_as(C.POINTER(C.c_int64)),
                                         k.ctypes.data_as(C.POINTER(C.c_int64)), out.ctypes.data_as(C.c_void_p)))
    rng = RRandom(7, kind)
    want = sum((rng.sample_int(int(a), int(b)) for a, b in zip(n, k)), [])
    assert out.tolist() == want
    assert out[:5].tolist() != sorted(out[:5].tolist()) or len(set(out[:5])) == 5


def test_duplicate_rows_redraw_from_unique_when_nstart_is_1():
    x = np.repeat(np.arange(6, dtype=np.float64)[:, None], 5, axis=0)      # 30 rows, 6 distinct
    for seed in range(1, 200):
        first = np.array(RRandom(seed).sample_int(30, 3)) - 1
        if len(set(x[first, 0])) < 3:
            break
    rows = K.initial_centres(x, 3, 1, seed)
    rng = RRandom(seed)
    rng.sample_int(30, 3)                                   # the first draw, discarded
    cn = K.unique_rows(x)
    assert rows[0].tolist() == cn[np.array(rng.sample_int(cn.shape[0], 3)) - 1].tolist()
    assert len(set(x[rows[0], 0])) == 3


def test_draws_of_several_starts():
    x = np.arange(40, dtype=np.float64).reshape(20, 2)
    rows = K.initial_centres(x, 4, 3, 42)
    rng = RRandom(42)
    assert rows.tolist() == [(np.array(rng.sample_int(20, 4)) - 1).tolist() for _ in range(3)]


def test_unique_first_occurrence_and_signed_zero():
    x = np.array([[1.0, 0.0], [2.0, 3.0], [1.0, -0.0], [2.0, 3.0], [0.0, 0.0], [-0.0, 0.0], [5.0, 1.0]])
    assert K.unique_rows(x).tolist() == [0, 1, 4, 6]


def test_fewer_distinct_rows_than_k():
    x = np.zeros((10, 3))
    x[5:] = 1.0
    with pytest.raises(K.KmeansError, match="more cluster centers than distinct data points"):
        K.kmeans(x, 3, nstart=2)


# ---------------------------------------------------------------- oracle properties ----------
def blobs(m, p, k, seed, spread=1.0):
    rng = np.random.default_rng(seed)
    c = rng.normal(0, 6, size=(k, p))
    lab = rng.integers(0, k, size=m)
    return np.asfortranarray(c[lab] + rng.normal(0, spread, size=(m, p)))


def sqd(x, c):
    return ((x[:, None, :] - c[None, :, :]) ** 2).sum(axis=2)


@pytest.mark.parametrize("alg", ["Lloyd", "MacQueen"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_lloyd_and_macqueen_end_at_a_fixed_point(alg, seed):
    x = blobs(300, 4, 4, seed)
    z = K.kmeans(x, 4, iter_max=50, nstart=3, algorithm=alg, seed=seed)
    assert z["ifault"] == 0
    cl = z["cluster"] - 1
    d = sqd(x, z["centers"])
    assert np.all(d[np.arange(x.shape[0]), cl] <= d.min(axis=1) * (1 + 1e-12))
    for l in range(4):
        np.testing.assert_allclose(z["centers"][l], x[cl == l].mean(axis=0), rtol=1e-12, atol=1e-12)
    assert z["size"].tolist() == np.bincount(cl, minlength=4).tolist()


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_hartigan_wong_ends_hartigan_optimal(seed):
    x = blobs(250, 3, 5, seed, spread=3.0)
    z = K.kmeans(x, 5, iter_max=50, nstart=2, seed=seed)
    if z["ifault"] in (2, 4):
        pytest.skip("stopped early")
    cl = z["cluster"] - 1
    n = np.bincount(cl, minlength=5).astype(np.float64)
    d = sqd(x, z["centers"])
    for i in range(x.shape[0]):
        l1 = cl[i]
        if n[l1] <= 1:
            continue
        lose = n[l1] / (n[l1] - 1) * d[i, l1]
        for l in range(5):
            if l != l1:
                assert n[l] / (n[l] + 1) * d[i, l] >= lose * (1 - 1e-9)
    np.testing.assert_allclose(z["withinss"].sum(), d[np.arange(x.shape[0]), cl].sum(), rtol=1e-12)


@pytest.mark.parametrize("alg", ALGS)
def test_hand_solved(alg):
    x = np.array([[0.0, 0.0], [0.0, 1.0], [10.0, 0.0], [10.0, 1.0], [0.0, 0.5], [10.0, 0.5]])
    z = K.kmeans(x, 2, nstart=4, algorithm=alg, seed=3)
    cl = z["cluster"]
    assert cl[0] == cl[1] == cl[4] and cl[2] == cl[3] == cl[5] and cl[0] != cl[2]
    left = cl[0] - 1
    np.testing.assert_array_equal(z["centers"][left], [0.0, 0.5])
    np.testing.assert_array_equal(z["centers"][1 - left], [10.0, 0.5])
    np.testing.assert_allclose(z["withinss"], [0.5, 0.5])
    np.testing.assert_allclose(z["totss"], 151.0)


def test_k_one_is_the_mean():
    x = blobs(50, 3, 2, 9)
    z = K.kmeans(x, 1, algorithm="Hartigan-Wong")
    assert z["cluster"].tolist() == [1] * 50 and z["iter"] == 1
    np.testing.assert_allclose(z["centers"][0], x.mean(axis=0), rtol=1e-13)


# ---------------------------------------------------------------- kmeansDesign host logic ----
class _Recorder:
    def __init__(self):
        self.calls = []

    def __call__(self, x, centers, iter_max=10, nstart=1, algorithm="Hartigan-Wong", seed=42, **kw):
        self.calls.append(dict(x=np.array(x), k=centers, iter_max=iter_max, nstart=nstart, algorithm=algorithm,
                               seed=seed, rownames=getattr(x, "rownames", None)))
        z = K.kmeans(np.asarray(x), centers, iter_max, nstart, algorithm, seed)
        return z


@pytest.fixture
def recorder(monkeypatch):
    from recoup_b200 import consumers
    r = _Recorder()
    monkeypatch.setattr(consumers, "kmeans", r)
    return r


def _input():
    from recoup_b200.profile import ProfileMatrix
    a = ProfileMatrix(blobs(40, 3, 3, 1), rownames=["g%d" % i for i in range(40)])
    b = ProfileMatrix(blobs(40, 2, 3, 2), rownames=["g%d" % i for i in range(40)])
    return [dict(id="WT", profile=a), dict(id="KO", profile=b)]


def test_kmeans_design_k0_returns_design(recorder):
    import recoup_b200 as rb
    d = {"Treatment": np.array(["a"] * 40)}
    assert rb.kmeansDesign(_input(), d) is d
    assert rb.kmeansDesign(_input(), None, dict(k=0)) is None
    assert recorder.calls == []


def test_kmeans_design_cbind_defaults_and_labels(recorder):
    import recoup_b200 as rb
    inp = _input()
    out = rb.kmeansDesign(inp, None, dict(k=3))
    c = recorder.calls[-1]
    np.testing.assert_array_equal(c["x"], np.hstack([inp[0]["profile"], inp[1]["profile"]]))
    assert (c["k"], c["nstart"], c["iter_max"], c["algorithm"], c["seed"]) == (3, 20, 20, "Hartigan-Wong", 42)
    assert c["rownames"] == inp[0]["profile"].rownames
    z = K.kmeans(c["x"], 3, 20, 20)
    assert out["Cluster"].tolist() == ["Cluster %d" % v for v in z["cluster"]]


def test_kmeans_design_reference_and_existing_design(recorder):
    import recoup_b200 as rb
    inp = _input()
    d = {"Treatment": np.array(["t%d" % (i % 2) for i in range(40)])}
    out = rb.kmeansDesign(inp, d, dict(k=2, reference="KO", nstart=3, algorithm="Lloyd", iterMax=7, seed=5))
    c = recorder.calls[-1]
    np.testing.assert_array_equal(c["x"], inp[1]["profile"])
    assert (c["nstart"], c["iter_max"], c["algorithm"], c["seed"]) == (3, 7, "Lloyd", 5)
    assert list(out) == ["Treatment", "Cluster"] and "Cluster" not in d
    assert out["Treatment"] is d["Treatment"]


def test_kmeans_design_unknown_reference_warns_and_uses_all(recorder):
    import recoup_b200 as rb
    inp = _input()
    with pytest.warns(UserWarning, match="reference nope not found"):
        rb.kmeansDesign(inp, None, dict(k=2, reference="nope"))
    assert recorder.calls[-1]["x"].shape == (40, 5)


def test_kmeans_argument_checks_before_the_device():
    import recoup_b200 as rb
    with pytest.raises(ValueError, match="should be one of"):
        rb.kmeans(np.zeros((4, 2)), 2, algorithm="Ward")
    with pytest.raises(TypeError):
        rb.kmeans(np.zeros((4, 2)), np.zeros((2, 2)))
    from recoup_b200.consumers import _match_algorithm
    assert _match_algorithm("Forgy") == "Forgy" and _match_algorithm("Mac") == "MacQueen"
    assert _match_algorithm(["Lloyd", "MacQueen"]) == "Lloyd"


# ---------------------------------------------------------------- on the device --------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import recoup_b200 as rb
    rb.init(0)
    return rb


def fixture_c1_profiles():
    from oracle import recoup_oracle as O
    from tests.helpers import fixture_genes, fixture_reads
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "recoup_test_data.npz"))
    genes, _ = fixture_genes(z)
    bp = dict(flankBinSize=0, regionBinSize=100, sumStat="mean", interpolation="auto")
    mats = []
    for s in (0, 1):
        reads, _ = fixture_reads(z, s)
        cov = O.coverage_ref(reads, genes, "tss", (2000, 2000))
        mats.append(O.profile_matrix(cov, (2000, 2000), bp))
    return np.asfortranarray(np.hstack(mats))


def gamma_zeros_dups(seed=5):
    rng = np.random.default_rng(seed)
    x = np.round(rng.gamma(0.8, 2.0, size=(600, 12)), 1)
    x[rng.random(size=x.shape) < 0.3] = 0.0
    x[rng.random(600) < 0.15] = 0.0                       # whole zero rows
    dup = rng.integers(0, 600, size=120)
    x[rng.integers(0, 600, size=120)] = x[dup]
    return np.asfortranarray(x)


INPUTS = {
    "blobs": lambda: blobs(800, 6, 5, 11),
    "gamma": gamma_zeros_dups,
    "c1": fixture_c1_profiles,
    "rows1e5": lambda: blobs(100_000, 4, 6, 12, spread=2.5),
    "p3000": lambda: blobs(120, 3000, 4, 13, spread=40.0),
}
_CACHE = {}


def get_input(name):
    if name not in _CACHE:
        _CACHE[name] = INPUTS[name]()
    return _CACHE[name]


def assert_matches_oracle(got, want):
    """Every field bit for bit against the start R keeps; when the device kept another start, that
    start's sum(wss) must tie the oracle's within 1e-12 (a tie R's long-double sum() may break either
    way, DESIGN.md section 2) and the device result must equal that start bit for bit."""
    best = want["best"]
    cands = [best] + [s for s in range(len(want["starts"])) if s != best and
                      abs(want["tots"][s] - want["tots"][best]) <= 1e-12 * abs(want["tots"][best])]
    for s in cands:
        w = want["starts"][s]
        if (np.array_equal(np.asarray(got["cluster"]), w["cluster"]) and got["size"].tolist() == w["size"].tolist()
                and got["iter"] == w["iter"] and got["ifault"] == w["ifault"]
                and np.array_equal(got["centers"], w["centers"], equal_nan=True)):
            np.testing.assert_allclose(got["withinss"], w["withinss"], rtol=1e-12, atol=1e-300)
            np.testing.assert_allclose(got["totss"], want["totss"], rtol=1e-12)
            return
    w = want["starts"][best]
    np.testing.assert_array_equal(np.asarray(got["cluster"]), w["cluster"])
    assert got["size"].tolist() == w["size"].tolist()
    assert (got["iter"], got["ifault"]) == (w["iter"], w["ifault"])
    np.testing.assert_array_equal(got["centers"], w["centers"])


@gpu
@pytest.mark.parametrize("name", list(INPUTS))
@pytest.mark.parametrize("nstart", [1, 20])
@pytest.mark.parametrize("k", [1, 2, 5, 17])
@pytest.mark.parametrize("alg", ALGS)
def test_device_equals_oracle(rb, alg, k, nstart, name):
    x = get_input(name)
    iter_max = 20
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            want = K.kmeans(x, k, iter_max, nstart, alg, seed=42, all_starts=True)
        except K.KmeansError as e:
            with pytest.raises(rb.RecoupError) as ei:
                rb.kmeans(x, k, iter_max, nstart, alg)
            assert str(e) in str(ei.value)
            return
        got = rb.kmeans(x, k, iter_max, nstart, alg)
    assert_matches_oracle(got, want)


@gpu
@pytest.mark.parametrize("alg", ALGS)
def test_host_and_device_memory_agree(rb, alg):
    import torch
    from recoup_b200 import _lib
    x = gamma_zeros_dups(7)
    want = rb.kmeans(x, 4, 20, 5, alg)
    m, p = x.shape
    xd = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()          # column-major on the device
    cl = torch.empty(m, dtype=torch.int32, device="cuda")
    cen = torch.empty((p, 4), dtype=torch.float64, device="cuda")    # k x p column-major
    wss = torch.empty(4, dtype=torch.float64, device="cuda")
    size = torch.empty(4, dtype=torch.int32, device="cuda")
    tot, it, fault, warn = C.c_double(), C.c_int(), C.c_int(), C.c_int()
    torch.cuda.synchronize()
    _lib.check(_lib.lib.rcp_kmeans(C.c_void_p(xd.data_ptr()), m, p, m, 4, 5, 20, {"Hartigan-Wong": 1, "Lloyd": 2,
                                   "MacQueen": 3}[alg], 42, 0, _lib.MEM_DEVICE, C.c_void_p(cl.data_ptr()),
                                   C.c_void_p(cen.data_ptr()), C.c_void_p(wss.data_ptr()),
                                   C.c_void_p(size.data_ptr()), C.byref(tot), C.byref(it), C.byref(fault),
                                   C.byref(warn)))
    _lib.check(_lib.lib.rcp_sync())
    np.testing.assert_array_equal(cl.cpu().numpy(), np.asarray(want["cluster"]))
    np.testing.assert_array_equal(cen.cpu().numpy().T, want["centers"])
    np.testing.assert_array_equal(wss.cpu().numpy(), want["withinss"])
    np.testing.assert_array_equal(size.cpu().numpy(), want["size"])
    assert (tot.value, it.value, fault.value) == (want["totss"], want["iter"], want["ifault"])


def _code(rb, fn):
    with pytest.raises(rb.RecoupError) as ei:
        fn()
    return ei.value.code, str(ei.value)


@gpu
def test_errors(rb):
    from recoup_b200 import _lib
    x = blobs(30, 3, 3, 1)
    for kw in (dict(centers=0), dict(centers=3, nstart=0), dict(centers=3, iter_max=0), dict(centers=31)):
        assert _code(rb, lambda: rb.kmeans(x, **kw))[0] == _lib.RCP_ERR_ARG
    assert "more cluster centers than data points" in _code(rb, lambda: rb.kmeans(x, 31))[1]
    out = np.zeros(40)
    i32 = np.zeros(40, np.int32)
    rc = _lib.lib.rcp_kmeans(x.ctypes.data_as(C.c_void_p), 30, 3, 30, 3, 1, 10, 7, 42, 0, 0,
                             i32.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                             out.ctypes.data_as(C.c_void_p), i32.ctypes.data_as(C.c_void_p), C.byref(C.c_double()),
                             C.byref(C.c_int()), C.byref(C.c_int()), C.byref(C.c_int()))
    assert rc == _lib.RCP_ERR_ARG
    bad = x.copy()
    bad[7, 2] = np.nan
    code, msg = _code(rb, lambda: rb.kmeans(bad, 3))
    assert code == _lib.RCP_ERR_DATA and "NA/NaN/Inf in foreign function call" in msg
    bad[7, 2] = np.inf
    assert _code(rb, lambda: rb.kmeans(bad, 3))[0] == _lib.RCP_ERR_DATA
    few = np.zeros((10, 2))
    few[5:] = 1.0
    code, msg = _code(rb, lambda: rb.kmeans(few, 3, nstart=2))
    assert code == _lib.RCP_ERR_DATA and "more cluster centers than distinct data points." in msg
    sq = np.arange(10, dtype=np.float64).reshape(5, 2)
    code, msg = _code(rb, lambda: rb.kmeans(sq, 5, nstart=2))
    assert code == _lib.RCP_ERR_DATA and "must lie between 1 and nrow(x)" in msg
    # two distinct rows whose squared distance underflows to 0: the later centre loses every tie and
    # is empty after the first assignment (kmns IFAULT = 1)
    tiny = np.array([[0.0], [1e-200], [7.0]])
    seed = next(s for s in range(1, 500) if sorted(np.array(RRandom(s).sample_int(3, 2)) - 1) == [0, 1])
    with pytest.raises(K.KmeansError, match="empty cluster"):
        K.kmeans(tiny, 2, seed=seed)
    code, msg = _code(rb, lambda: rb.kmeans(tiny, 2, seed=seed))
    assert code == _lib.RCP_ERR_DATA and "empty cluster: try a better set of initial centers" in msg


@gpu
@pytest.mark.parametrize("alg", ALGS)
def test_iter_max_1_does_not_converge(rb, alg):
    x = blobs(2000, 3, 6, 21, spread=4.0)
    want = K.kmeans(x, 6, 1, 1, alg, all_starts=True)
    with pytest.warns(UserWarning, match="did not converge in 1 iteration$"):
        got = rb.kmeans(x, 6, iter_max=1, algorithm=alg)
    assert got["ifault"] == 2 and got["iter"] == 2
    assert_matches_oracle(got, want)


@gpu
def test_kmeans_design_on_device_profiles(rb):
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
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = rb.kmeansDesign(inp, None, dict(k=4, nstart=5))
        want = K.kmeans(np.hstack([np.asarray(s["profile"]) for s in inp]), 4, 20, 5, all_starts=True)
        got = rb.kmeans(rb.ProfileMatrix(np.hstack([np.asarray(s["profile"]) for s in inp]),
                                         rownames=inp[0]["profile"].rownames), 4, 20, 5)
    assert_matches_oracle(got, want)
    assert out["Cluster"].tolist() == ["Cluster %d" % c for c in got["cluster"]]
    assert got["cluster"].names == inp[0]["profile"].rownames
    ref = rb.kmeansDesign(inp, None, dict(k=3, reference="KO", nstart=4))
    assert ref["Cluster"].shape[0] == len(inp[1]["profile"])
