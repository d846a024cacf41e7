"""Distributional cores on the GPU (agents/core_distributional.py twins) vs the reference's numba goldens and vs the
C oracle on fresh seeded arenas (including the low-visit random pick through the injected RNG stream)."""
import os

import numpy as np
import pytest

from arena_gen import golden_bk_dist, make_dist_arena

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "dist_golden.npz")


def test_dist_twins_match_reference_golden(gpu_lib):
    from tetris_mcts_b200.agents import core_distributional as CD
    z = np.load(GOLD)
    for i in range(int(z["n_cases"])):
        p = "d%d_" % i
        assert np.allclose(CD.shift_distribution(z[p + "dist"], float(z[p + "x"]), 0, 5000), z[p + "shift"], rtol=1e-5, atol=1e-7)
        assert np.allclose(CD.mean_variance(z[p + "dist"], 0, 5000), z[p + "mv"], rtol=1e-5)
        tr = CD.select_trace_distributional(1, z[p + "child"], z[p + "node_stats"], z[p + "node_dist"], 0, 5000, low=0)
        assert np.array_equal(tr, z[p + "trace"]), i
        ns, nd = z[p + "node_stats"].copy(), z[p + "node_dist"].copy()
        CD.backup_trace_distributional(z[p + "trace"], ns, nd, float(z[p + "r"]), z[p + "dist"], 0, 5000)
        assert np.allclose(ns, z[p + "bk_stats"], rtol=1e-5, atol=1e-5)
        assert np.allclose(nd, golden_bk_dist(z, p), rtol=1e-5, atol=1e-7)


def test_dist_twins_match_oracle_with_rng(gpu_lib, oracle):
    from tetris_mcts_b200.agents import core_distributional as CD
    rng = np.random.default_rng(1)
    for seed in range(6):
        a = make_dist_arena(50 + seed, M=512, max_depth=6, unvisited=0.25)
        for low in (0, 1, 5):
            CD.rng_state[0] = 777 + seed
            st = np.array([777 + seed], np.uint32)
            got = CD.select_trace_distributional(1, a["child"], a["node_stats"], a["node_dist"], 0, 5000, low=low)
            want = oracle.select_trace_distributional(1, a["child"], a["node_stats"], low, rng_state=st)
            assert np.array_equal(got, want) and CD.rng_state[0] == st[0]
        dist = rng.random(50).astype(np.float32)
        dist /= dist.sum()
        ns1, nd1, ns2, nd2 = a["node_stats"].copy(), a["node_dist"].copy(), a["node_stats"].copy(), a["node_dist"].copy()
        r = float(a["node_stats"][want[-1], 2] + 40)
        CD.backup_trace_distributional(want, ns1, nd1, r, dist, 0, 5000)
        oracle.backup_trace_distributional(want, ns2, nd2, r, dist, 0, 5000)
        assert np.array_equal(ns1, ns2) and np.array_equal(nd1, nd2)


def _search_seed(seed, g):
    s = (seed + 0x9E3779B9 * (g + 1)) & 0xffffffff
    return s or 0x2545F491


def test_dist_engine_matches_oracle_agent(gpu_lib, oracle):
    """BASELINE config 5 path end to end (select_trace_distributional -> evaluate leaf -> expand -> backup_trace_distributional),
    synthetic histogram evaluator on both sides: actions, stats and the node_stats / node_dist arrays must be identical."""
    from tetris_mcts_b200 import pyTetris as PT
    from tetris_mcts_b200.engine import BatchedEngine
    n, M, sims, moves, seed = 12, 4096, 60, 10, 77
    recs = PT.new_games(n, (1, 0, 0), np.arange(seed, seed + n, dtype=np.uint32))
    eng = BatchedEngine(n, max_nodes=M, mode="dist", eval_kind="synthetic", seed=seed)
    eng.set_games(recs)
    agents = [oracle.Agent(max_nodes=M, mode=3, low=5, eval_mode=0, search_seed=_search_seed(seed, g)) for g in range(n)]
    games = [oracle.Game(record=recs[g]) for g in range(n)]
    for g in range(n):
        agents[g].update_root(games[g].record())
    for mv in range(moves):
        eng.run_sims(sims)
        stats, action = eng.get_stats()
        for g in range(n):
            agents[g].mcts(sims)
            a, st = agents[g].get_action()
            assert np.array_equal(st, stats[g]), (mv, g, st, stats[g])
            assert a == action[g]
            games[g].play(a)
            agents[g].update_root(games[g].record())
            if games[g].end:
                games[g].reset()
                agents[g].update_root(games[g].record())
        eng.env_step(None)
        eng.update_root(auto_reset=True)
    for g in range(4):
        ns, nd = eng.export_dist(g)
        wns, wnd = agents[g].export_dist()
        assert np.array_equal(ns, wns) and np.array_equal(nd, wnd), g
    eng.close()


@pytest.mark.parametrize("kind", ["net", "net_tc"])
def test_dist_network_matches_reference_golden(gpu_lib, oracle, kind):
    """model/model_distributional.py Net (torch CPU) outputs recorded in tests/golden/distnet_golden.npz; fp32 CUDA cores ("net") and the
    tcgen05 path ("net_tc": fp16 x 2 operand split, north_star's 1e-5 on the probabilities)."""
    from tetris_mcts_b200.engine import BatchedEngine
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "distnet_golden.npz"))
    w = oracle.seeded_dist_weights(int(z["seed"]))
    eng = BatchedEngine(1, max_nodes=64, mode="dist", eval_kind=kind, dist_weights=w)
    got = eng.distnet(z["states"])
    atol = 1e-7 if kind == "net" else 1e-6
    assert np.allclose(got, z["dist"], rtol=1e-5, atol=atol), np.abs(got - z["dist"]).max()
    assert np.allclose(got, oracle.distnet_forward(w, z["states"]), rtol=1e-5, atol=atol)
    assert np.allclose(got.sum(axis=1), 1.0, atol=1e-5)
    eng.close()


def test_dist_network_tensor_core_path_matches_cuda_core_path(gpu_lib, oracle):
    """Every batch size from one board to several 128-board tiles per CTA, position-independent."""
    from arena_gen import boards
    from tetris_mcts_b200.engine import BatchedEngine
    w = oracle.seeded_dist_weights(3)
    et = BatchedEngine(1, max_nodes=64, mode="dist", eval_kind="net_tc", dist_weights=w)
    es = BatchedEngine(1, max_nodes=64, mode="dist", eval_kind="net", dist_weights=w)
    for n in (1, 2, 3, 5, 127, 129, 700, 20000):
        s = boards(n, n)
        a, b = et.distnet(s), es.distnet(s)
        assert np.allclose(a, b, rtol=1e-5, atol=1e-6), (n, np.abs(a - b).max())
        if n == 700:
            assert np.array_equal(et.distnet(s[::-1])[::-1], a)
    et.close(); es.close()


@pytest.mark.parametrize("kind", ["net", "net_tc"])
def test_dist_engine_runs_with_network(gpu_lib, oracle, kind):
    from tetris_mcts_b200 import pyTetris as PT
    from tetris_mcts_b200.engine import BatchedEngine
    n = 256
    eng = BatchedEngine(n, max_nodes=2048, mode="dist", eval_kind=kind, dist_weights=oracle.seeded_dist_weights(0), overflow_reset=True)
    eng.set_games(PT.new_games(n, (1, 0, 0), np.arange(1, n + 1, dtype=np.uint32)))
    for _ in range(3):
        actions, stats = eng.play_move(100, auto_reset=True)
    ns, nd = eng.export_dist(0)
    live = ns[:, 0] > 0
    assert live.any() and np.allclose(nd[live].sum(axis=1), 1.0, atol=1e-3)
    assert eng.counters()["sims"] == n * 300
    eng.close()
