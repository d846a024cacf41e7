"""Oracle parity AT THE BENCHMARKED CONFIGURATION (BASELINE configs[2] as bench.py runs it): 16384 games, max_nodes 16384, 500 simulations
per move, the tcgen05 network (eval net_tc), set_gc_headroom(2560), overflow_reset, the production path (one CUDA graph per simulation
step, b200_play_move).  The C oracle agent cannot shadow 16384 games, so a sample of them is shadowed game for game: the oracle agents are fed
the GPU network's outputs for the same boards (the LP search is deterministic given evaluator and piece sequence, SURVEY N3), make the same
remove_nodes() calls the head-room policy makes (agents/agent.py:246-257 driven as in tests/golden/gen_golden.py gen_agent_explicit_gc) and
apply the same overflow_reset rule (oracle/mcts_oracle.c drop_tree).  Compared exactly: action and stats[3,7] of every move
(agents/agent.py:153-185), the live games, and the exported arenas in the reference's array layout (agents/agent.py:58-88), with the
path cache on (the default at this configuration) and off.
Reference loop: agents/ValueSimLP.py:44-70."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ARGS = (1, 0, 0)


def search_seed(seed, g):
    s = (seed + 0x9E3779B9 * (g + 1)) & 0xffffffff
    return s or 0x2545F491


@pytest.mark.parametrize("path_cache", [True, False], ids=["cache_on", "cache_off"])
def test_bench_config_sampled_games_exact(gpu_lib, oracle, path_cache):
    from tetris_mcts_b200 import pyTetris as PT
    from tetris_mcts_b200.engine import BatchedEngine
    from tetris_mcts_b200.model.model_vv import init_weights
    n, M, sims, moves, headroom, seed = 16384, 16384, 500, 14, 16384 * 5 // 32, 123
    recs = PT.new_games(n, ARGS, np.arange(seed, seed + n, dtype=np.uint32))
    w = init_weights(0)
    eng = BatchedEngine(n, max_nodes=M, mode="lp", eval_kind="net_tc", weights=w, seed=seed, overflow_reset=True, path_cache=path_cache)
    assert eng.path_cache == path_cache
    eng.set_games(recs)
    eng.set_gc_headroom(headroom)
    side = BatchedEngine(1, max_nodes=64, eval_kind="net_tc", weights=w)

    def cb(states):
        return side.valuenet(states)

    sample = sorted(set([0, n - 1] + list(np.random.default_rng(7).choice(n, 14, replace=False))))
    agents = {g: oracle.Agent(max_nodes=M, mode=0, gamma=0.999, low=1, eval_mode=2, eval_cb=cb, search_seed=search_seed(seed, g),
                              overflow_reset=1) for g in sample}
    games = {g: oracle.Game(record=recs[g]) for g in sample}
    for g in sample:
        agents[g].update_root(games[g].record())
    for mv in range(moves):
        actions, stats = eng.play_move(sims, auto_reset=True)                 # graph replay, get_action, play, update_root, head-room collection
        live = eng.get_games()
        for g in sample:
            agents[g].mcts(sims)
            a, st = agents[g].get_action()
            assert a == actions[g] and np.array_equal(st, stats[g]), "move %d game %d\n%s\n%s" % (mv, g, st, stats[g])
            games[g].play(a)
            agents[g].update_root(games[g].record())
            if games[g].end:
                games[g].reset()
                agents[g].update_root(games[g].record())
            if agents[g].n_free < headroom:
                agents[g].remove_nodes()
            assert np.array_equal(live[g], games[g].record()), "live game %d differs after move %d" % (g, mv)
    c = eng.counters()
    assert c["sims"] == n * sims * moves and (eng.status() == 0).all()
    assert c["gcs"] > 0, "the window must contain collections"
    sampled_gcs = sum(agents[g].counter(3) for g in sample)
    assert sampled_gcs > 0, "no sampled game collected: lengthen the window"
    for g in sample:
        ex, want = eng.export_game(g), agents[g].export()
        assert ex["root"] == agents[g].root, g
        for k in ("child", "n2o", "episode", "score", "visit", "value", "variance", "obs_end", "obs_key", "game"):
            assert np.array_equal(ex[k], want[k]), (g, k)
    print("bench-config parity: %d sampled games x %d moves exact; collections %d (sampled %d), trees dropped %d (sampled %d), mean trace %.1f"
          % (len(sample), moves, c["gcs"], sampled_gcs, c["tree_resets"], sum(agents[g].counter(7) for g in sample),
             c["trace_levels"] / c["sims"]))
    side.close()
    eng.close()


def test_overflow_reset_rule_matches_oracle_small(gpu_lib, oracle):
    """The same shadowing with arenas so small that trees are dropped all the time (inside expansions, inside update_root and by the
    head-room collection): the engine's overflow_reset (k_gc + reset_tree) against oracle/mcts_oracle.c drop_tree, every move, every game."""
    from tetris_mcts_b200 import pyTetris as PT
    from tetris_mcts_b200.engine import BatchedEngine
    n, M, sims, moves, headroom, seed = 48, 512, 40, 40, 200, 31
    recs = PT.new_games(n, ARGS, np.arange(seed, seed + n, dtype=np.uint32))
    for hr in (headroom, 0):
        eng = BatchedEngine(n, max_nodes=M, mode="lp", eval_kind="synthetic", seed=seed, overflow_reset=True)
        eng.set_games(recs)
        eng.set_gc_headroom(hr)
        agents = [oracle.Agent(max_nodes=M, mode=0, gamma=0.999, low=1, eval_mode=0, search_seed=search_seed(seed, g), overflow_reset=1) for g in range(n)]
        games = [oracle.Game(record=recs[g]) for g in range(n)]
        for g in range(n):
            agents[g].update_root(games[g].record())
        for mv in range(moves):
            actions, stats = eng.play_move(sims, auto_reset=True)
            for g in range(n):
                agents[g].mcts(sims)
                a, st = agents[g].get_action()
                assert a == actions[g] and np.array_equal(st, stats[g]), (hr, mv, g)
                games[g].play(a)
                agents[g].update_root(games[g].record())
                if games[g].end:
                    games[g].reset()
                    agents[g].update_root(games[g].record())
                if hr and agents[g].n_free < hr:
                    agents[g].remove_nodes()
        c = eng.counters()
        assert c["tree_resets"] == sum(ag.counter(7) for ag in agents) > 0
        assert c["gcs"] == sum(ag.counter(3) for ag in agents)
        assert c["expansions"] == sum(ag.counter(1) for ag in agents)
        for g in (0, n // 2, n - 1):
            ex, want = eng.export_game(g), agents[g].export()
            for k in ("child", "n2o", "episode", "score", "visit", "value", "variance", "obs_end", "obs_key", "game"):
                assert np.array_equal(ex[k], want[k]), (hr, g, k)
        eng.close()
