"""calcDesignPlotProfiles: the per-level curves of a design-split profile plot.  The per-level
restatement (plot_design_profiles, built on oracle.recoup_oracle.plot_profile) against a
brute-force loop and the host logic of calcDesignPlotProfiles on
the CPU; rcp_matrix_group_col_profile against the oracle and against colProfile of each level's
rows under `-m gpu` on a B200."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import recoup_oracle as O


# ---------------------------------------------------------------- per-level restatement ------
def plot_design_profiles(profile, design, avgfun="mean", scale="natural"):
    """calcDesignPlotProfiles without smoothing, PARITY UNPINNED (the reference's source of it is
    not in this image; the level rules are this library's contract): O.plot_profile over the rows
    of every level of `design`, a dict of equal-length label columns in row order.  A level is the
    label of the single column, or the tuple of labels across columns; only combinations that
    occur are levels, ordered by each column's sorted labels (factor()), first column slowest; a
    row with a None label is in no level.  Returns [(level, rows (1-based), plot_profile)]."""
    cols = [list(v) for v in design.values()]
    n = len(cols[0])
    keep = [i for i in range(n) if all(c[i] is not None for c in cols)]
    sorted_labels = [sorted({c[i] for i in keep}) for c in cols]
    key = {i: tuple(sorted_labels[j].index(cols[j][i]) for j in range(len(cols))) for i in keep}
    x = np.asarray(profile, dtype=np.float64)
    out = []
    for k in sorted(set(key.values())):
        rows = [i for i in keep if key[i] == k]
        labels = tuple(sorted_labels[j][k[j]] for j in range(len(cols)))
        level = labels[0] if len(cols) == 1 else labels
        out.append((level, np.array(rows) + 1, O.plot_profile(x[rows], avgfun, scale)))
    return out


# ---------------------------------------------------------------- oracle on the CPU -----------
def brute_levels(design):
    """Level -> 0-based rows by a loop over every label combination of the sorted columns."""
    import itertools
    cols = list(design.values())
    n = len(cols[0])
    uniq = [sorted({v for v in c if v is not None}) for c in cols]
    out = []
    for combo in itertools.product(*uniq):
        rows = [i for i in range(n) if all(cols[j][i] == combo[j] for j in range(len(cols)))]
        if rows:
            out.append((combo[0] if len(cols) == 1 else combo, rows))
    return out


def brute_profile(x, avgfun, scale):
    x = np.log2(x + 1.0) if scale == "log2" else x
    if avgfun == "mean":
        c = np.array([float(np.mean(x[:, j].astype(np.longdouble))) for j in range(x.shape[1])])
        s = np.array([float(np.std(x[:, j].astype(np.longdouble), ddof=1)) if x.shape[0] > 1 else np.nan
                      for j in range(x.shape[1])])
    else:
        c = np.median(x, axis=0)
        s = 1.4826 * np.median(np.abs(x - c), axis=0)
    return c, s


def test_oracle_equals_brute_force_per_level():
    rng = np.random.default_rng(1)
    x = np.round(rng.gamma(0.7, 2.0, size=(40, 6)), 1)
    a = [None if i == 7 else "L%d" % (i % 4) for i in range(40)]
    a[11] = "solo"                                   # a one-row level
    b = ["+" if i % 3 else "-" for i in range(40)]
    b[20] = None
    for design in ({"a": a}, {"a": a, "b": b}, {"b": b}):
        for avgfun in ("mean", "median"):
            for scale in ("natural", "log2"):
                got = plot_design_profiles(x, design, avgfun, scale)
                want = brute_levels(design)
                assert [lv for lv, _, _ in got] == [lv for lv, _ in want]
                for (lv, rows, prof), (_, wrows) in zip(got, want):
                    assert rows.tolist() == [r + 1 for r in wrows]
                    c, s = brute_profile(x[wrows], avgfun, scale)
                    np.testing.assert_allclose(prof["profile"], c, rtol=1e-13)
                    np.testing.assert_allclose(prof["upper"], c + s, rtol=1e-13, equal_nan=True)


# ---------------------------------------------------------------- calcDesignPlotProfiles (host)
@pytest.fixture
def oracle_groups(monkeypatch):
    """calcDesignPlotProfiles with the oracle standing in for the device call; records the codes."""
    from recoup_b200 import consumers
    seen = []

    def fake(mats, codes, n_groups, avgfun, log2):
        seen.append((np.array(codes), n_groups))
        out = []
        for m in mats:
            cen = np.full((n_groups, m.shape[1]), np.nan)
            spr = np.full((n_groups, m.shape[1]), np.nan)
            for g in range(n_groups):
                rows = np.flatnonzero(codes == g + 1)
                p = O.plot_profile(m[rows], avgfun, "log2" if log2 else "natural")
                cen[g] = p["profile"]
                spr[g] = p["upper"] - p["profile"]
            out.append((cen, spr))
        return out
    monkeypatch.setattr(consumers, "_group_profiles", fake)
    return seen


def _inp(n=30, seed=3):
    rng = np.random.default_rng(seed)
    return [{"id": "A", "profile": rng.integers(0, 5, size=(n, 4)).astype(float)},
            {"id": "B", "profile": rng.integers(0, 5, size=(n, 7)).astype(float)}]


OPTS = {"plotParams": {"sumStat": "mean", "signalScale": "natural", "smooth": False}}


def _check_against_oracle(got, inp, design, avgfun="mean", scale="natural"):
    for s, x in enumerate(inp):
        want = plot_design_profiles(x["profile"], design, avgfun, scale)
        assert [lv for lv, _, _ in got] == [lv for lv, _, _ in want]
        for (lv, rows, curves), (_, wrows, wprof) in zip(got, want):
            assert rows.dtype == np.int32 and rows.tolist() == wrows.tolist()
            assert len(curves) == len(inp)
            for k in ("profile", "upper", "lower"):
                np.testing.assert_allclose(curves[s][k], wprof[k], rtol=1e-12, atol=1e-12, equal_nan=True)


def test_levels_sort_as_factor_does(oracle_groups):
    from recoup_b200 import calcDesignPlotProfiles
    inp = _inp()
    lab = ["Cluster %d" % (1 + i % 11) for i in range(30)]
    got = calcDesignPlotProfiles(inp, {"Cluster": lab}, OPTS)
    levels = [lv for lv, _, _ in got]
    assert levels == sorted(set(lab))
    assert levels.index("Cluster 10") < levels.index("Cluster 2")
    for lv, rows, _ in got:
        assert rows.tolist() == [i + 1 for i in range(30) if lab[i] == lv]
    _check_against_oracle(got, inp, {"Cluster": lab})
    codes, g = oracle_groups[-1]
    assert g == 11 and codes.min() == 1 and codes.max() == 11


def test_tuple_levels_and_excluded_rows(oracle_groups):
    from recoup_b200 import calcDesignPlotProfiles
    inp = _inp()
    strand = ["+" if i < 12 else "-" for i in range(30)]
    clus = ["k%d" % (i % 3) for i in range(30)]
    for i in range(12):                              # ("+", "k2") never occurs
        if clus[i] == "k2":
            clus[i] = "k0"
    clus[4] = None
    strand[25] = None
    design = {"strand": strand, "Cluster": clus}
    got = calcDesignPlotProfiles(inp, design, OPTS)
    assert [lv for lv, _, _ in got] == [("+", "k0"), ("+", "k1"), ("-", "k0"), ("-", "k1"), ("-", "k2")]
    all_rows = np.concatenate([rows for _, rows, _ in got])
    assert 5 not in all_rows and 26 not in all_rows and all_rows.shape[0] == 28
    codes, g = oracle_groups[-1]
    assert g == 5 and codes[4] == 0 and codes[25] == 0
    _check_against_oracle(got, inp, design)
    opts = {"plotParams": {"sumStat": "median", "signalScale": "log2"}}
    _check_against_oracle(calcDesignPlotProfiles(inp, design, opts), inp, design, "median", "log2")


def test_design_errors(oracle_groups):
    from recoup_b200 import calcDesignPlotProfiles
    inp = _inp()
    with pytest.raises(ValueError, match="design column Cluster has 29 rows"):
        calcDesignPlotProfiles(inp, {"Cluster": ["a"] * 29}, OPTS)
    for bad in ({}, None):
        with pytest.raises(ValueError, match="at least one column"):
            calcDesignPlotProfiles(inp, bad, OPTS)
    with pytest.raises(NotImplementedError):
        calcDesignPlotProfiles(inp, {"Cluster": ["a"] * 30}, {"plotParams": {"smooth": True}})
    assert oracle_groups == []


def test_kmeans_design_used_directly(oracle_groups, monkeypatch):
    from recoup_b200 import calcDesignPlotProfiles, consumers, kmeansDesign
    inp = _inp()

    def fake_kmeans(x, centers, **kw):
        return {"cluster": np.array([1 + (i * 7) % centers for i in range(x.shape[0])], dtype=np.int32)}
    monkeypatch.setattr(consumers, "kmeans", fake_kmeans)
    design = kmeansDesign(inp, None, {"k": 3})
    got = calcDesignPlotProfiles(inp, design, OPTS)
    assert [lv for lv, _, _ in got] == ["Cluster 1", "Cluster 2", "Cluster 3"]
    _check_against_oracle(got, inp, design)


# ---------------------------------------------------------------- on the device --------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import recoup_b200 as rb
    rb.init(0)
    return rb


def bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    """equal bit for bit, any NaN equal to any NaN and -0.0 to 0.0 (the keys of the sort order them as equal)"""
    a, b = np.asarray(a, dtype=np.float64) + 0.0, np.asarray(b, dtype=np.float64) + 0.0
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(np.where(na, 0.0, a)), bits(np.where(nb, 0.0, b)))


def oracle_groups_of(x, codes, G, avgfun, scale, groups):
    """the oracle's profile, upper and lower of every level in `groups` (NaN elsewhere)"""
    out = np.full((3, G, x.shape[1]), np.nan)
    for g in groups:
        rows = np.flatnonzero(codes == g + 1)
        if rows.shape[0]:
            p = O.plot_profile(x[rows], avgfun, scale)
            out[:, g] = p["profile"], p["upper"], p["lower"]
    return out


def check_groups(rb, x, codes, G, avgfun, scale, exact_mean=False):
    cen, spr = rb.groupColProfile(x, codes, G, avgfun, scale)
    assert cen.shape == (G, x.shape[1]) and spr.shape == (G, x.shape[1])
    check = range(G) if G <= 64 else sorted(np.random.default_rng(G).choice(G, size=64, replace=False).tolist())
    wc, wu, wl = oracle_groups_of(x, codes, G, avgfun, scale, check)
    for g in check:
        rows = np.flatnonzero(codes == g + 1)
        if rows.shape[0] == 0:
            assert np.all(np.isnan(cen[g])) and np.all(np.isnan(spr[g])), g
            continue
        sc, ss = rb.colProfile(np.asfortranarray(x[rows]), avgfun, scale)
        if avgfun == "median" and scale == "natural":
            assert same_bits(cen[g], wc[g]) and same_bits(cen[g] + spr[g], wu[g]), g
            assert same_bits(cen[g] - spr[g], wl[g]), g
        if avgfun == "median":
            # log2 on the device and in numpy may differ in the last bit, so on that scale the
            # bit-for-bit reference is the library's own one-group call on the level's rows
            assert same_bits(cen[g], sc) and same_bits(spr[g], ss), g
        if avgfun == "mean" or scale == "log2":
            for got, want in ((cen[g], wc[g]), (cen[g] + spr[g], wu[g]), (cen[g] - spr[g], wl[g])):
                np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12, equal_nan=True)
        if avgfun == "mean":
            if exact_mean:
                assert same_bits(cen[g], sc) and same_bits(spr[g], ss), g
            if rows.shape[0] == 1:
                assert np.all(np.isnan(spr[g]))
        if avgfun == "median" and rows.shape[0] == 1:
            assert np.all((spr[g] == 0) | np.isnan(x[rows[0]]))
    return cen, spr


def _matrices():
    rng = np.random.default_rng(77)
    a = rng.gamma(0.6, 3.0, size=(2001, 37))
    a[rng.random(a.shape) < 0.3] = 0.0                    # many ties at zero
    a[5] = 0.0
    b = np.round(rng.normal(0.0, 2.0, size=(64, 5)), 1)   # negatives, ties, -0.0
    b[3, 2] = -0.0
    b[7, 1] = -0.0
    ints = rng.integers(0, 6, size=(900, 9)).astype(float)
    return {"gamma": a, "signed": b, "one_row": rng.random((1, 4)), "one_col": rng.random((700, 1)), "ints": ints}


def _codes(n, G, rng, exclude=False):
    codes = (np.arange(n) % G + 1).astype(np.int32)       # interleaved, as k-means labels come
    codes = codes[rng.permutation(n)] if G < n else codes
    if exclude and n > 3:
        codes[rng.integers(0, n, size=max(1, n // 10))] = 0
        codes[0] = -3
        codes[n // 2] = np.iinfo(np.int32).min
    return codes


@gpu
@pytest.mark.parametrize("avgfun", ["mean", "median"])
@pytest.mark.parametrize("scale", ["natural", "log2"])
def test_device_equals_oracle(rb, avgfun, scale):
    rng = np.random.default_rng(5)
    for name, x in _matrices().items():
        if scale == "log2" and x.min() < 0:
            continue
        x = np.asfortranarray(x)
        n = x.shape[0]
        for G in sorted({1, 2, 5, 64, n}):
            for exclude in (False, True):
                codes = _codes(n, G, rng, exclude)
                check_groups(rb, x, codes, G, avgfun, scale, exact_mean=(name == "ints"))
        # empty groups: codes only reach 3 of 7
        check_groups(rb, x, _codes(n, 3, rng), 7, avgfun, scale, exact_mean=(name == "ints"))


@gpu
@pytest.mark.parametrize("avgfun", ["mean", "median"])
def test_one_row_per_group_is_the_matrix(rb, avgfun):
    x = np.asfortranarray(_matrices()["gamma"][:500])
    n = x.shape[0]
    codes = np.random.default_rng(9).permutation(n).astype(np.int32) + 1
    for scale in ("natural", "log2"):
        cen, spr = rb.groupColProfile(x, codes, n, avgfun, scale)
        if scale == "natural":
            assert same_bits(cen[codes - 1], x)
        else:
            # log2 on the device and in numpy may differ in the last bit: the scaled matrix is
            # the one-row call's result, and within two units in the last place of numpy's
            np.testing.assert_array_max_ulp(cen[codes - 1], np.log2(x + 1.0), maxulp=2)
            for r in np.random.default_rng(10).choice(n, size=20, replace=False):
                assert same_bits(cen[codes[r] - 1], rb.colProfile(x[[r]], avgfun, scale)[0]), r
        if avgfun == "mean":
            assert np.all(np.isnan(spr))
        else:
            assert np.all(spr == 0)
    cen, spr = rb.groupColProfile(x, None, 1, avgfun)
    want_c, want_s = rb.colProfile(x, avgfun)
    assert same_bits(cen[0], want_c) and same_bits(spr[0], want_s)


def _abi(m_ptr, n, p, ld, codes_ptr, G, stat, lg, mem, c_ptr, s_ptr):
    from recoup_b200 import _lib
    return _lib.lib.rcp_matrix_group_col_profile(m_ptr, n, p, ld, codes_ptr, G, stat, lg, mem, c_ptr, s_ptr)


vp = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731


@gpu
def test_row_block_of_taller_matrix_and_device_memory(rb):
    import torch
    from recoup_b200 import _lib
    rng = np.random.default_rng(12)
    tall = np.asfortranarray(np.round(rng.gamma(0.8, 2.0, size=(1300, 30)), 1))
    n, p, G = 1000, 30, 6
    codes = _codes(n, G, rng, exclude=True)
    for stat, avgfun in ((0, "mean"), (1, "median")):
        want = rb.groupColProfile(np.asfortranarray(tall[:n]), codes, G, avgfun, "log2")
        cen = np.empty((G, p), order="F")
        spr = np.empty((G, p), order="F")
        _lib.check(_abi(vp(tall), n, p, tall.shape[0], vp(codes), G, stat, 1, _lib.MEM_HOST, vp(cen), vp(spr)))
        assert same_bits(cen, want[0]) and same_bits(spr, want[1])
        xd = torch.from_numpy(np.ascontiguousarray(tall.T)).cuda()
        cd = torch.from_numpy(codes).cuda()
        co = torch.empty((p, G), dtype=torch.float64, device="cuda")
        so = torch.empty_like(co)
        torch.cuda.synchronize()
        _lib.check(_abi(C.c_void_p(xd.data_ptr()), n, p, tall.shape[0], C.c_void_p(cd.data_ptr()), G, stat, 1,
                        _lib.MEM_DEVICE, C.c_void_p(co.data_ptr()), C.c_void_p(so.data_ptr())))
        _lib.check(_lib.lib.rcp_sync())
        assert same_bits(co.cpu().numpy().T, want[0]) and same_bits(so.cpu().numpy().T, want[1])
        again = rb.groupColProfile(np.asfortranarray(tall[:n]), codes, G, avgfun, "log2")
        assert same_bits(again[0], want[0]) and same_bits(again[1], want[1])


@gpu
@pytest.mark.parametrize("avgfun", ["mean", "median"])
def test_large_matrix(rb, avgfun):
    rng = np.random.default_rng(21)
    n, p = 200_000, 400
    x = np.asfortranarray(rng.gamma(0.6, 3.0, size=(n, p)))
    x[rng.random(n) < 0.2] = 0.0
    for G, sample in ((5, None), (20_000, 40)):
        codes = _codes(n, G, rng)
        cen, spr = rb.groupColProfile(x, codes, G, avgfun)
        levels = range(G) if sample is None else sorted(rng.choice(G, size=sample, replace=False).tolist())
        for g in levels:
            rows = np.flatnonzero(codes == g + 1)
            want = O.plot_profile(x[rows], avgfun)
            if avgfun == "median":
                assert same_bits(cen[g], want["profile"]), g
                assert same_bits(cen[g] + spr[g], want["upper"]), g
            else:
                np.testing.assert_allclose(cen[g], want["profile"], rtol=1e-12)
                np.testing.assert_allclose(cen[g] + spr[g], want["upper"], rtol=1e-12)


def pool_used():
    from tests.test_hclust import pool_used as pu
    return pu()


@gpu
def test_errors_leave_no_memory_behind(rb):
    from recoup_b200 import _lib
    x = np.zeros(64)
    codes = np.ones(64, np.int32)
    out = np.zeros(4096)
    out2 = np.zeros(4096)

    def code(n, p, ld, G=2, stat=0, mem=_lib.MEM_HOST, cds=codes, c_out=out, s_out=out2, xx=x):
        _lib.check(_lib.lib.rcp_sync())
        before = pool_used()
        rc = _abi(vp(xx) if xx is not None else None, n, p, ld, vp(cds) if cds is not None else None, G, stat, 0, mem,
                  vp(c_out) if c_out is not None else None, vp(s_out) if s_out is not None else None)
        msg = _lib.lib.rcp_last_error().decode()
        _lib.check(_lib.lib.rcp_sync())
        assert pool_used() == before, (n, p, msg)
        return rc, msg

    assert code(8, 4, 7)[0] == _lib.RCP_ERR_ARG                      # ld < n_rows
    assert code(-1, 4, 8)[0] == _lib.RCP_ERR_ARG
    assert code(8, 4, 8, mem=5)[0] == _lib.RCP_ERR_ARG
    assert code(8, 4, 8, stat=2) == (_lib.RCP_ERR_ARG, "col_profile: bad stat")
    assert code(8, 4, 8, G=0)[0] == _lib.RCP_ERR_ARG
    assert code(8, 4, 8, c_out=None) == (_lib.RCP_ERR_ARG, "col_profile: NULL output")
    assert code(0, 4, 1) == (_lib.RCP_ERR_ARG, "col_profile: the matrix has no rows")
    assert code(8, 4, 8, xx=None)[0] == _lib.RCP_ERR_ARG
    big = code(1 << 20, 1 << 12, 1 << 20, mem=_lib.MEM_DEVICE, cds=None, c_out=out, s_out=out2)
    assert big[0] == _lib.RCP_ERR_UNSUPPORTED, big
    assert code(10, 1 << 20, 10, G=1 << 12, mem=_lib.MEM_DEVICE)[0] == _lib.RCP_ERR_UNSUPPORTED
    bad = codes.copy()
    bad[13] = 3
    for stat in (0, 1):
        rc, msg = code(16, 4, 16, G=2, stat=stat, cds=bad)
        assert rc == _lib.RCP_ERR_DATA and "greater than n_groups" in msg
    assert code(16, 4, 16, G=2)[0] == _lib.RCP_OK
    assert code(16, 4, 16, G=2, cds=None)[0] == _lib.RCP_OK


def _fixture_input(rb):
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
    strand_of = dict(zip([str(g) for g in z["gene_names"]], z["gene_strand"].tolist()))
    return inp, strand_of


@gpu
def test_end_to_end_on_the_fixture(rb):
    inp, strand_of = _fixture_input(rb)
    design = rb.kmeansDesign(inp, None, {"k": 3})
    names = inp[0]["profile"].rownames
    n = np.asarray(inp[0]["profile"]).shape[0]
    if names is not None:
        strand = ["+" if strand_of[str(r)] > 0 else "-" for r in names]
    else:
        strand = ["+" if s > 0 else "-" for s in list(strand_of.values())[:n]]
    for d in ({"Cluster": design["Cluster"]}, {"strand": strand, "Cluster": design["Cluster"]}):
        for avgfun in ("mean", "median"):
            opts = {"plotParams": {"sumStat": avgfun, "signalScale": "natural"}}
            got = rb.calcDesignPlotProfiles(inp, d, opts)
            assert len(got) >= 3
            _check_against_oracle(got, inp, d, avgfun)
