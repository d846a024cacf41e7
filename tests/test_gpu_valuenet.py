"""Value network forward (model/model_vv.py:13-52, :210-217) on the GPU vs the C oracle and vs golden outputs of
the reference's own Model_VV (torch CPU).  Tolerance from north_star: 1e-5 (relative, fp32)."""
import os

import numpy as np
import pytest

from arena_gen import boards

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "valuenet_golden.npz")
RTOL, ATOL = 1e-5, 1e-5


def _boards_unused(n, seed):
    """tools/test.py:23-28 style boards: random {0,1}, top rows cleared, four -1 cells; plus real game positions."""
    rng = np.random.default_rng(seed)
    b = (rng.random((n, 20, 10)) < 0.45).astype(np.int8)
    for i in range(n):
        b[i, :rng.integers(2, 12)] = 0
        r, c = rng.integers(0, 3), rng.integers(0, 8)
        b[i, r:r + 2, c:c + 2] = -1
    return b


@pytest.mark.parametrize("kind", ["net", "net_tc"])
def test_matches_oracle(gpu_lib, oracle, kind):
    from tetris_mcts_b200.engine import BatchedEngine
    w = oracle.seeded_weights(0)
    eng = BatchedEngine(1, max_nodes=64, eval_kind=kind, weights=w)
    for n in (1, 3, 4, 7, 64, 250, 1000):
        s = boards(n, n)
        v, var = eng.valuenet(s)
        wv, wvar = oracle.valuenet_forward(w, s)
        assert np.allclose(v, wv, rtol=RTOL, atol=ATOL), np.abs(v - wv).max()
        assert np.allclose(var, wvar, rtol=RTOL, atol=ATOL), np.abs(var - wvar).max()
    eng.close()


@pytest.mark.parametrize("kind", ["net", "net_tc"])
def test_batch_position_independent(gpu_lib, oracle, kind):
    """The same board must give the same bits wherever it sits in the batch (search determinism relies on it)."""
    from tetris_mcts_b200.engine import BatchedEngine
    eng = BatchedEngine(1, max_nodes=64, eval_kind=kind, weights=oracle.seeded_weights(1))
    s = boards(300, 9)
    v1, r1 = eng.valuenet(s)
    perm = np.random.default_rng(0).permutation(300)
    v2, r2 = eng.valuenet(s[perm])
    assert np.array_equal(v1[perm], v2) and np.array_equal(r1[perm], r2)
    eng.close()


@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden vectors not generated")
@pytest.mark.parametrize("kind", ["net", "net_tc"])
def test_matches_reference_golden(gpu_lib, oracle, kind):
    from tetris_mcts_b200.engine import BatchedEngine
    z = np.load(GOLD)
    for seed in z["seeds"]:
        w = oracle.seeded_weights(int(seed))
        eng = BatchedEngine(1, max_nodes=64, eval_kind=kind, weights=w)
        v, var = eng.valuenet(z["states"])
        assert np.allclose(v, z["v_%d" % seed], rtol=RTOL, atol=ATOL), np.abs(v - z["v_%d" % seed]).max()
        assert np.allclose(var, z["var_%d" % seed], rtol=RTOL, atol=ATOL), np.abs(var - z["var_%d" % seed]).max()
        eng.close()


def test_tensor_core_path_matches_cuda_core_path(gpu_lib, oracle):
    """Every batch size from one board to two or three 128-board FC tiles per CTA (40000 boards = 313 tiles), position-independent."""
    from tetris_mcts_b200.engine import BatchedEngine
    w = oracle.seeded_weights(3)
    et = BatchedEngine(1, max_nodes=64, eval_kind="net_tc", weights=w)
    es = BatchedEngine(1, max_nodes=64, eval_kind="net", weights=w)
    for n in (1, 129, 700, 20000, 40000):
        s = boards(n, n)
        (vt, rt), (vs, rs) = et.valuenet(s), es.valuenet(s)
        assert np.allclose(vt, vs, rtol=RTOL, atol=ATOL), (n, np.abs(vt - vs).max())
        assert np.allclose(rt, rs, rtol=RTOL, atol=ATOL), (n, np.abs(rt - rs).max())
        if n == 700:
            v2, r2 = et.valuenet(s[::-1])
            assert np.array_equal(v2[::-1], vt) and np.array_equal(r2[::-1], rt)
    et.close(); es.close()


def test_tensor_core_conv_stack_matches_cuda_core_path(gpu_lib, oracle):
    """Layer-level check of the tcgen05 shift-GEMM convolutions: the flatten input of fc1 from both device paths."""
    import ctypes as C
    from tetris_mcts_b200.engine import BatchedEngine
    from tetris_mcts_b200 import _lib as L
    w = oracle.seeded_weights(2)
    s = np.ascontiguousarray(boards(37, 5).reshape(-1, 200))
    outs = {}
    for kind in ("net", "net_tc"):
        eng = BatchedEngine(1, max_nodes=64, eval_kind=kind, weights=w)
        o = np.zeros((len(s), 1792), np.float32)
        L.check(L.lib().b200_debug_act3(eng.h, L.ptr(s), len(s), L.ptr(o)))
        outs[kind] = o
        eng.close()
    assert np.abs(outs["net"]).max() > 0.01
    assert np.allclose(outs["net"], outs["net_tc"], rtol=2e-6, atol=2e-6), np.abs(outs["net"] - outs["net_tc"]).max()
