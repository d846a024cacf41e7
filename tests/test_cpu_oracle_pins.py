"""Pin the CPU oracle (oracle/*.c) to the reference: against the committed golden vectors that were produced by
running the reference itself (tests/golden/gen_golden.py), on stored inputs and on seeded arenas regenerated here."""
import os

import numpy as np

from arena_gen import arena_crc, make_arena, near_tie_arena, state_to_obskey

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_core_golden(oracle):
    z = np.load(os.path.join(GOLD, "core_golden.npz"))
    for i in range(int(z["n_cases"])):
        p = "c%d_" % i
        a = {k: z[p + k] for k in ("child", "visit", "value", "variance", "score", "n2o")}
        tr = oracle.select_trace_obs(1, a["child"], a["visit"], a["value"], a["variance"], a["score"], a["n2o"], int(z[p + "low"]),
                                     rng_state=np.array([1], np.uint32))
        assert np.array_equal(tr, z[p + "trace"])
        cn, co = oracle.get_unique_child_obs(int(z[p + "uniq_node"]), a["child"], a["score"], a["n2o"])
        assert np.array_equal(cn, z[p + "uniq_c"]) and np.array_equal(co, z[p + "uniq_o"])
        b = {k: a[k].copy() for k in ("visit", "value", "variance")}
        oracle.backup_trace_obs(tr, b["visit"], b["value"], b["variance"], a["n2o"], a["score"], float(z[p + "bk_v"]),
                                float(z[p + "bk_var"]), float(z[p + "gamma"]))
        for k in b:
            assert np.array_equal(b[k], z[p + "bk_" + k]), (i, k)
        for m in (0, 1):
            for av in (0, 1):
                b = {k: a[k].copy() for k in ("visit", "value", "variance")}
                oracle.backup_trace_obs_LP(z[p + "lp_trace"], b["visit"], b["value"], b["variance"], a["n2o"], a["score"], z[p + "lp_end"],
                                           z[p + "lp_c"], z[p + "lp_o"], z[p + "lp_v"], z[p + "lp_var"], float(z[p + "gamma"]), m, av)
                for k in b:
                    assert np.array_equal(b[k], z[p + "lp%d%d_" % (m, av) + k]), (i, m, av, k)
        assert oracle.get_all_childs(1, a["child"]) == set(z[p + "reach"].tolist())


def test_valuenet_golden(oracle):
    z = np.load(os.path.join(GOLD, "valuenet_golden.npz"))
    for seed in z["seeds"]:
        v, var = oracle.valuenet_forward(oracle.seeded_weights(int(seed)), z["states"])
        assert np.allclose(v, z["v_%d" % seed], rtol=1e-5, atol=1e-5)
        assert np.allclose(var, z["var_%d" % seed], rtol=1e-5, atol=1e-5)


def test_agent_golden(oracle):
    """The C agent vs the reference's own Python ValueSimLP + agent.py + compiled core.cpp (exact)."""
    z = np.load(os.path.join(GOLD, "agent_golden.npz"))
    for case in range(int(z["n_cases"])):
        p = "a%d_" % case
        ag = oracle.Agent(max_nodes=int(z[p + "M"]), mode=0, gamma=0.999, low=1, eval_mode=0)
        g = oracle.Game(record=z[p + "start"])
        ag.update_root(g.record())
        for mv, act in enumerate(z[p + "actions"]):
            ag.mcts(int(z[p + "sims"]))
            a, st = ag.get_action()
            assert a == act and np.array_equal(st, z[p + "stats"][mv]), (case, mv)
            g.play(a)
            ag.update_root(g.record())
            if g.end:
                g.reset()
                ag.update_root(g.record())
        ex = ag.export()
        for k in ("child", "score", "n2o", "visit", "value", "variance", "episode"):
            assert np.array_equal(ex[k], z[p + k]), (case, k)
        assert ag.root == int(z[p + "root"])
        if case == 1:
            assert ag.counter(3) > 0, "the GC case must collect garbage"


def test_agent_explicit_remove_nodes_golden(oracle):
    """TreeAgent.remove_nodes() called by the driver between moves (agents/agent.py:246-257 is a public method): the C agent
    with the same calls vs the reference's own ValueSimLP (tests/golden/gen_golden.py: gen_agent_explicit_gc).  This is the
    collection policy the engine batches over all games (b200_set_gc_headroom / b200_remove_nodes)."""
    z = np.load(os.path.join(GOLD, "agent_gc_golden.npz"))
    for case in range(int(z["n_cases"])):
        p = "g%d_" % case
        ag = oracle.Agent(max_nodes=int(z[p + "M"]), mode=0, gamma=0.999, low=1, eval_mode=0)
        g = oracle.Game(record=z[p + "start"])
        ag.update_root(g.record())
        collected = []
        for mv, act in enumerate(z[p + "actions"]):
            ag.mcts(int(z[p + "sims"]))
            a, st = ag.get_action()
            assert a == act and np.array_equal(st, z[p + "stats"][mv]), (case, mv)
            g.play(a)
            ag.update_root(g.record())
            if g.end:
                g.reset()
                ag.update_root(g.record())
            if ag.n_free < int(z[p + "headroom"]):
                ag.remove_nodes()
                collected.append(mv)
        assert np.array_equal(np.array(collected, np.int32), z[p + "collected"])
        assert ag.n_free == int(z[p + "n_free"])
        ex = ag.export()
        for k in ("child", "score", "n2o", "visit", "value", "variance", "episode"):
            assert np.array_equal(ex[k], z[p + k]), (case, k)
        assert ag.root == int(z[p + "root"])


def test_agent_modes_golden(oracle):
    """The other two mcts loops: the C agent in MODE_SINGLE / MODE_VANILLA vs the reference's own agents/ValueSim.py and
    agents/Vanilla.py, whose rand() (check_low, core.h:62,76) and randint (Vanilla.py:52) were served from the oracle's xorshift
    stream when the golden was generated (oracle/rand_shim.c, gen_agent_modes) — exact, including a case with collections."""
    z = np.load(os.path.join(GOLD, "agent_modes_golden.npz"))
    for case in range(int(z["n_cases"])):
        p = "m%d_" % case
        mode = int(z[p + "mode"])
        ag = oracle.Agent(max_nodes=int(z[p + "M"]), mode=mode, gamma=0.999 if mode == 1 else 0.99, low=1 if mode == 1 else 5,
                          eval_mode=0, search_seed=int(z[p + "search_seed"]))
        g = oracle.Game(record=z[p + "start"])
        ag.update_root(g.record())
        for mv, act in enumerate(z[p + "actions"]):
            ag.mcts(int(z[p + "sims"]))
            a, st = ag.get_action()
            assert a == act and np.array_equal(st, z[p + "stats"][mv]), (case, mv)
            g.play(a)
            ag.update_root(g.record())
            if g.end:
                g.reset()
                ag.update_root(g.record())
        ex = ag.export()
        for k in ("child", "score", "n2o", "visit", "value", "variance", "episode"):
            assert np.array_equal(ex[k], z[p + k]), (case, k)
        assert ag.root == int(z[p + "root"])
        if case == 1:
            assert ag.counter(5) > 1000, "the Vanilla case must roll out"
        if case == 2:
            assert ag.counter(3) > 0, "the small-arena case must collect garbage"


def test_agent_cpp_golden(oracle):
    """The reference's C++ agent twin (agents/cppmodule/agent.cpp, compiled unchanged, leaf-parallel MCTSAgent) vs the C agent with
    lp_end_from_obs=1 (agent.cpp:538) and lp_var_gamma2=0 (agent.cpp:558): the flags the engine exposes for that behaviour
    (SURVEY N1).  The module exposes play() only: the action and the game record after every move must agree."""
    z = np.load(os.path.join(GOLD, "agent_cpp_golden.npz"))
    for case in range(int(z["n_cases"])):
        p = "c%d_" % case
        ag = oracle.Agent(max_nodes=100000, mode=0, gamma=0.999, low=1, eval_mode=0, lp_end_from_obs=1, lp_var_gamma2=0)
        g = oracle.Game(record=z[p + "start"])
        ag.update_root(g.record())
        for mv, act in enumerate(z[p + "actions"]):
            ag.mcts(int(z[p + "sims"]))
            a, _ = ag.get_action()
            assert a == act, (case, mv)
            g.play(a)
            assert np.array_equal(g.record(), z[p + "records"][mv]), (case, mv)
            ag.update_root(g.record())
            if g.end:
                g.reset()
                ag.update_root(g.record())
    # the Python-path flags give a different game on the same seed: the golden does discriminate between the two variants
    ag = oracle.Agent(max_nodes=100000, mode=0, gamma=0.999, low=1, eval_mode=0)
    g = oracle.Game(record=z["c1_start"])
    ag.update_root(g.record())
    same = True
    for mv, act in enumerate(z["c1_actions"]):
        ag.mcts(int(z["c1_sims"]))
        a, _ = ag.get_action()
        if a != act:
            same = False
            break
        g.play(a)
        ag.update_root(g.record())
        if g.end:
            g.reset()
            ag.update_root(g.record())
    assert not same


def test_env_spec_examples(oracle):
    """Hand-checkable rules of SPEC_PYTETRIS.md §2-4."""
    g = oracle.Game(1, 0, 0, seed=7)
    s = g.state()
    assert (s == -1).sum() == 4 and (s == 1).sum() == 0 and (s[:2] == -1).sum() == 4      # spawn in rows 0-1
    g.play(5)                                                                               # hard drop
    s = g.state()
    assert (s[18:] == 1).sum() >= 2 and g.score > 0                                         # locked at the bottom, 2 pts/row
    g2 = oracle.Game(1, 1, 0, seed=7)
    g2.play(5)
    assert g2.score == 0                                                                    # scoring=1 counts lines only
    # 7-bag: the first seven pieces are a permutation
    g = oracle.Game(1, 0, 0, seed=99)
    seen = []
    for _ in range(7):
        seen.append(int(g.record()[10]) & 7)
        g.play(5)
    assert sorted(seen) == list(range(7))
    # line clear: fill the bottom row except the columns an I piece covers, then drop the I
    rec = oracle.Game(1, 0, 0, seed=1).record()
    rec[9] = np.uint32((0x3ff & ~(0xf << 3)) << 16)          # row 19 full except cols 3-6
    rec[10] = (rec[10] & ~np.uint32(0x3fff)) | np.uint32(0 | (0 << 3) | ((3 + 2) << 5) | ((-1 + 2) << 9))   # I piece, spawn pose
    g = oracle.Game(record=rec)
    g.play(5)
    assert g.line_clears == 1 and g.score == 2 * 19 + 100 and int(g.record()[15]) == 1 and (g.state() == 1).sum() == 0


def test_synthetic_eval_is_plain_integer_hash(oracle):
    s = np.zeros((20, 10), np.int8)
    s[19, :5] = 1
    s[0, 3:7] = -1
    v, var = oracle.synthetic_eval(state_to_obskey(s))
    assert 0 <= v < 64 and 0.5 <= var < 64.5 and v * 256 == int(v * 256) and (var - 0.5) * 16 == int((var - 0.5) * 16)


def test_live_against_reference_core(oracle):
    """select_trace_obs / backup_trace_obs on 30 seeded arenas vs what the reference's own compiled core.cpp returned on them
    (tests/golden/gen_golden.py gen_core_live): the arenas are regenerated here, the golden holds their CRC-32 and the reference's
    outputs.  The backed-up arrays must equal the reference's at the entries it changed and the input everywhere else."""
    z = np.load(os.path.join(GOLD, "core_live_golden.npz"))
    assert int(z["n_cases"]) == 30
    for seed in range(30):
        p = "s%d_" % seed
        a = make_arena(1000 + seed, M=1024, max_depth=4 + seed % 7) if seed % 5 else near_tie_arena(seed)
        assert arena_crc(a) == int(z[p + "crc"]), "arena %d no longer matches the one the golden was recorded on" % seed
        mine = oracle.select_trace_obs(1, a["child"], a["visit"], a["value"], a["variance"], a["score"], a["n2o"], 1)
        assert np.array_equal(z[p + "trace"], mine), seed
        b2 = {k: a[k].copy() for k in ("visit", "value", "variance")}
        oracle.backup_trace_obs(mine, b2["visit"], b2["value"], b2["variance"], a["n2o"], a["score"], 123.456, 7.89, 0.999)
        idx = z[p + "bk_idx"]
        for k in b2:
            want = a[k].copy()
            want[idx] = z[p + "bk_" + k]
            assert np.array_equal(want, b2[k]), (seed, k)
