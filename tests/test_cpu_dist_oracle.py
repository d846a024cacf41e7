"""Distributional cores (SURVEY §8a a16): the C oracle vs the reference's own numba functions (golden vectors; the
reference is compiled with fastmath, so floats are compared to 1e-5 relative, traces exactly)."""
import os

import numpy as np

from arena_gen import golden_bk_dist

GOLD = os.path.join(os.path.dirname(__file__), "golden", "dist_golden.npz")


def test_dist_oracle_matches_reference_numba(oracle):
    z = np.load(GOLD)
    for i in range(int(z["n_cases"])):
        p = "d%d_" % i
        assert np.allclose(oracle.shift_distribution(z[p + "dist"], float(z[p + "x"]), 0, 5000), z[p + "shift"], rtol=1e-5, atol=1e-7)
        m, v = oracle.mean_variance(z[p + "dist"], 0, 5000)
        assert np.allclose([m, v], z[p + "mv"], rtol=1e-5)
        tr = oracle.select_trace_distributional(1, z[p + "child"], z[p + "node_stats"], 0)
        assert np.array_equal(tr, z[p + "trace"]), i
        ns, nd = z[p + "node_stats"].copy(), z[p + "node_dist"].copy()
        oracle.backup_trace_distributional(z[p + "trace"], ns, nd, float(z[p + "r"]), z[p + "dist"], 0, 5000)
        assert np.allclose(ns, z[p + "bk_stats"], rtol=1e-5, atol=1e-5)
        assert np.allclose(nd, golden_bk_dist(z, p), rtol=1e-5, atol=1e-7)
