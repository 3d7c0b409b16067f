"""hclust parity against outputs of the REAL stats::hclust, when somebody has produced them.

`Rscript tools/make_r_golden.R` writes tests/golden/r_outputs/hclust_*: `hclust(dist(x))`
(complete linkage, Euclidean) of the C1 fixture profiles (both samples, cbind).  This module
compares the restatement (oracle/hclust_oracle.*) and, under `-m gpu`, rcp_hclust with them:
merge and order exactly, heights bit for bit (written with 17 significant digits).  Without that
directory the tests SKIP and hclust parity stays unpinned (DESIGN.md section 2).
"""
import os

import numpy as np
import pytest

from oracle import hclust_oracle as H

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "r_outputs")
needs_r = pytest.mark.skipif(not os.path.isfile(os.path.join(GOLD, "hclust_merge.csv")),
                             reason="no hclust outputs in tests/golden/r_outputs (run tools/make_r_golden.R "
                                    "with a real R): parity unpinned")


def r_result():
    merge = np.array([[int(v) for v in line.split(",")] for line in open(os.path.join(GOLD, "hclust_merge.csv"))])
    height = np.array([float(v) for v in open(os.path.join(GOLD, "hclust_height.txt")).read().split()])
    order = np.array([int(v) for v in open(os.path.join(GOLD, "hclust_order.txt")).read().split()])
    return dict(merge=merge, height=height, order=order)


def c1_matrix():
    from tests.test_kmeans import fixture_c1_profiles
    return fixture_c1_profiles()


def compare(got, want):
    np.testing.assert_array_equal(np.asarray(got["merge"]), want["merge"])
    np.testing.assert_array_equal(np.asarray(got["order"]), want["order"])
    np.testing.assert_array_equal(np.asarray(got["height"]), want["height"])


@needs_r
def test_oracle_against_r():
    compare(H.hclust(c1_matrix()), r_result())


@needs_r
@pytest.mark.gpu
def test_device_against_r():
    import recoup_b200 as rb
    rb.init(0)
    compare(rb.hclust(c1_matrix()), r_result())
