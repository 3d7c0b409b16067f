"""k-means parity against outputs of the REAL stats::kmeans, when somebody has produced them.

`Rscript tools/make_r_golden.R` writes tests/golden/r_outputs/kmeans_*: `set.seed(42); kmeans(x,
5, iter.max = 20, nstart, algorithm)` of the C1 fixture profiles (both samples, cbind), for every
algorithm and nstart in {1, 20}.  This module compares the restatement (oracle/kmeans_oracle.*)
and, under `-m gpu`, rcp_kmeans with them: cluster, centres and iter exactly, withinss within
1e-12.  Without that directory the tests SKIP and k-means parity stays unpinned (DESIGN.md
section 2).
"""
import os

import numpy as np
import pytest

from oracle import kmeans_oracle as K

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "r_outputs")
needs_r = pytest.mark.skipif(not os.path.isfile(os.path.join(GOLD, "kmeans_HartiganWong_nstart1_cluster.txt")),
                             reason="no k-means outputs in tests/golden/r_outputs (run tools/make_r_golden.R "
                                    "with a real R): parity unpinned")
ALGS = ["Hartigan-Wong", "Lloyd", "MacQueen"]


def r_result(alg, nstart):
    f = os.path.join(GOLD, "kmeans_%s_nstart%d_" % (alg.replace("-", ""), nstart))
    cluster = np.array([int(v) for v in open(f + "cluster.txt").read().split()])
    centers = np.array([[float(v) for v in line.split(",")] for line in open(f + "centers.csv")])
    withinss = np.array([float(v) for v in open(f + "withinss.txt").read().split()])
    it = int(open(f + "iter.txt").read().split()[0])
    return dict(cluster=cluster, centers=centers, withinss=withinss, iter=it)


def c1_matrix():
    from tests.test_kmeans import fixture_c1_profiles
    return fixture_c1_profiles()


def compare(got, want):
    np.testing.assert_array_equal(np.asarray(got["cluster"]), want["cluster"])
    np.testing.assert_array_equal(got["centers"], want["centers"])
    np.testing.assert_allclose(got["withinss"], want["withinss"], rtol=1e-12)
    assert got["iter"] == want["iter"]


@needs_r
@pytest.mark.parametrize("nstart", [1, 20])
@pytest.mark.parametrize("alg", ALGS)
def test_oracle_against_r(alg, nstart):
    compare(K.kmeans(c1_matrix(), 5, 20, nstart, alg, seed=42), r_result(alg, nstart))


@needs_r
@pytest.mark.gpu
@pytest.mark.parametrize("nstart", [1, 20])
@pytest.mark.parametrize("alg", ALGS)
def test_device_against_r(alg, nstart):
    import recoup_b200 as rb
    rb.init(0)
    compare(rb.kmeans(c1_matrix(), 5, 20, nstart, alg, seed=42), r_result(alg, nstart))
