"""Generate tests/golden/*.npz by RUNNING THE REFERENCE ITSELF in the build container (it cannot travel to the GPU box):
  core_golden.npz     outputs of the reference's own agents/cppmodule/core.cpp (compiled unchanged -> oracle/_ref/core*.so)
  core_live_golden.npz  the same core.cpp on 30 more arenas that tests/arena_gen.py regenerates from their seeds (only outputs stored)
  valuenet_golden.npz outputs of the reference's own model/model_vv.py Model_VV (torch CPU) with seeded weights
  dist_golden.npz     outputs of the reference's own numba cores agents/core_distributional.py (fastmath: pinned to 1e-5)
  agent_golden.npz    per-move statistics of the reference's own agents/ValueSimLP.py + agents/agent.py driving
                      the oracle env (the only non-reference part: pyTetris is absent upstream) with the synthetic
                      evaluator patched onto the agent instance (no reference file is modified)
  agent_gc_golden.npz the same agent with the driver calling agent.remove_nodes() between moves (public method)
  agent_cpp_golden.npz  actions / game records of the reference's own C++ agent twin (agents/cppmodule/agent.cpp compiled unchanged)
  agent_modes_golden.npz  the reference's own agents/ValueSim.py and agents/Vanilla.py (the other two mcts loops); their
                      rand() / randint draw from the oracle's xorshift stream (oracle/rand_shim.c, LD_PRELOAD)
  agent_online_golden.npz  the replay memory the reference's own OnlineMCTSAgent (agent.cpp, online) hands to its train callback under each of
                      its four accumulation policies (weighted / random trimming included), one process per policy
  train_golden.npz    optimiser steps of the reference's own Model_VV.train (model/model.py:95-119, GaussianLL model_vv.py:94-101,
                      Yogi model/yogi.py) on torch CPU; the torch-1.x overloads those files call are re-created at run time
Run:  python tests/golden/gen_golden.py      (needs /root/reference and `make -C oracle`)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import oracle_py as O  # noqa: E402
from arena_gen import arena_crc, make_arena, near_tie_arena, boards, state_to_obskey  # noqa: E402


def gen_core(core):
    out = {}
    cases = [dict(seed=s, M=1024, max_depth=4 + s % 6) for s in range(8)]
    cases += [dict(seed=20 + s, M=1024, max_depth=6, unvisited=0.3, single_low=True) for s in range(4)]
    rng = np.random.default_rng(0)
    for i, kw in enumerate(cases):
        a = make_arena(**kw)
        p = "c%d_" % i
        low = 1 if "unvisited" in kw else int(rng.choice([0, 1]))
        for k in ("child", "visit", "value", "variance", "score", "n2o"):
            out[p + k] = a[k]
        out[p + "low"] = low
        tr = core.select_trace_obs(1, a["child"], a["visit"], a["value"], a["variance"], a["score"], a["n2o"], low)
        out[p + "trace"] = np.asarray(tr, np.int32)
        un = int(tr[len(tr) // 2])
        c, o = core.get_unique_child_obs(un, a["child"], a["score"], a["n2o"])
        out[p + "uniq_node"], out[p + "uniq_c"], out[p + "uniq_o"] = un, np.asarray(c, np.int32), np.asarray(o, np.int32)
        v, var, gamma = float(rng.uniform(0, 400)), float(rng.uniform(0, 200)), float(rng.choice([0.999, 0.99]))
        out[p + "bk_v"], out[p + "bk_var"], out[p + "gamma"] = v, var, gamma
        b = {k: a[k].copy() for k in ("visit", "value", "variance")}
        core.backup_trace_obs(np.asarray(tr, np.int32), b["visit"], b["value"], b["variance"], a["n2o"], a["score"], v, var, gamma)
        for k in b:
            out[p + "bk_" + k] = b[k]
        lp_tr = np.asarray(tr[:-1] if len(tr) > 1 else tr, np.int32)
        c, o = core.get_unique_child_obs(int(lp_tr[-1]), a["child"], a["score"], a["n2o"])
        end = (rng.random(len(a["visit"])) < 0.1)
        lv = rng.uniform(0, 100, len(c)).astype(np.float32)
        lvar = rng.uniform(0.1, 1000, len(c)).astype(np.float32)
        out[p + "lp_trace"], out[p + "lp_c"], out[p + "lp_o"] = lp_tr, np.asarray(c, np.int32), np.asarray(o, np.int32)
        out[p + "lp_end"], out[p + "lp_v"], out[p + "lp_var"] = end.astype(np.uint8), lv, lvar
        for m in (0, 1):
            for av in (0, 1):
                b = {k: a[k].copy() for k in ("visit", "value", "variance")}
                core.backup_trace_obs_LP(lp_tr, b["visit"], b["value"], b["variance"], a["n2o"], a["score"], end, list(c), list(o), lv, lvar,
                                         gamma, bool(m), bool(av))
                for k in b:
                    out[p + "lp%d%d_" % (m, av) + k] = b[k]
        out[p + "reach"] = np.asarray(sorted(core.get_all_childs(1, a["child"])), np.int32)
    out["n_cases"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "core_golden.npz"), **out)
    print("core_golden: %d cases" % len(cases))


def gen_core_live(core):
    """core_live_golden.npz: select_trace_obs (low=1) and backup_trace_obs of the reference's own core.cpp on 30 arenas that
    tests/arena_gen.py regenerates from their seeds (every observation visited, so check_low never draws rand()).  The arenas
    are not stored, only their CRC-32; of the backed-up arrays only the entries the backup changed are stored (bk_idx)."""
    out = {}
    n = 30
    for seed in range(n):
        a = make_arena(1000 + seed, M=1024, max_depth=4 + seed % 7) if seed % 5 else near_tie_arena(seed)
        p = "s%d_" % seed
        tr = np.asarray(core.select_trace_obs(1, a["child"], a["visit"], a["value"], a["variance"], a["score"], a["n2o"], 1), np.int32)
        b = {k: a[k].copy() for k in ("visit", "value", "variance")}
        core.backup_trace_obs(tr, b["visit"], b["value"], b["variance"], a["n2o"], a["score"], 123.456, 7.89, 0.999)
        idx = np.nonzero(np.logical_or.reduce([b[k] != a[k] for k in b]))[0].astype(np.int32)
        out[p + "crc"], out[p + "trace"], out[p + "bk_idx"] = arena_crc(a), tr, idx
        for k in b:
            out[p + "bk_" + k] = b[k][idx]
    out["n_cases"] = n
    np.savez_compressed(os.path.join(HERE, "core_live_golden.npz"), **out)
    print("core_live_golden: %d cases" % n)


def gen_valuenet():
    import torch
    from model.model_vv import Model_VV
    torch.set_num_threads(1)
    states = np.concatenate([boards(48, 1), np.zeros((1, 20, 10), np.int8), -np.ones((1, 20, 10), np.int8) * 0 + 1])
    # real game positions too
    g = O.Game(seed=5)
    rng = np.random.default_rng(2)
    real = []
    while not g.end and len(real) < 14:
        g.play(int(rng.integers(0, 7)))
        real.append(g.state())
    states = np.concatenate([states, np.stack(real)]).astype(np.int8)
    out = dict(states=states, seeds=np.array([0, 1]))
    for seed in (0, 1):
        m = Model_VV(use_cuda=False)
        sd = {k: torch.from_numpy(v.copy()) for k, v in O.weights_to_state_dict(O.seeded_weights(seed)).items()}
        m.model.load_state_dict(sd)
        m.training(False)
        v, var = m.inference(states[:, None, :, :])
        out["v_%d" % seed], out["var_%d" % seed] = v.ravel().astype(np.float32), var.ravel().astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "valuenet_golden.npz"), **out)
    print("valuenet_golden: %d boards x 2 weight seeds" % len(states))


def synthetic_inference(batch):
    b = np.asarray(batch).reshape(-1, 20, 10)
    v = np.zeros((len(b), 1), np.float32)
    var = np.zeros((len(b), 1), np.float32)
    for i, s in enumerate(b):
        v[i, 0], var[i, 0] = O.synthetic_eval(state_to_obskey(s))
    return [v, var]


def gen_agent(pt):
    from agents.ValueSimLP import ValueSimLP
    out = {}
    cases = [dict(M=20000, sims=50, moves=20, seed=123), dict(M=2500, sims=40, moves=45, seed=321)]
    for i, cs in enumerate(cases):
        p = "a%d_" % i
        game = pt.Tetris((20, 10), 1, 0, 0)
        game.seed(cs["seed"])
        ag = ValueSimLP(sims=cs["sims"], env=pt.Tetris, env_args=((20, 10), 1, 0, 0), benchmark=False, online=False, min_visit=40)
        ag.max_nodes = cs["M"]          # public attribute + public method: the arena size is the only thing changed
        ag.init_array()
        ag.model.inference = synthetic_inference
        out[p + "start"] = np.array(game.get_record(), np.uint32)
        ag.update_root(game)
        acts, stats = [], []
        for mv in range(cs["moves"]):
            a = ag.play()
            acts.append(int(a))
            stats.append(ag.get_stats())
            game.play(a)
            ag.update_root(game)
            if game.end:
                game.reset()
                ag.update_root(game)
        out[p + "M"], out[p + "sims"] = cs["M"], cs["sims"]
        out[p + "actions"], out[p + "stats"] = np.array(acts, np.int32), np.stack(stats).astype(np.float32)
        for k in ("child", "score", "episode"):
            out[p + k] = ag.arrays[k]
        out[p + "n2o"] = ag.node_to_obs
        for k in ("visit", "value", "variance"):
            out[p + k] = ag.obs_arrays[k]
        out[p + "root"] = ag.root
    out["n_cases"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "agent_golden.npz"), **out)
    print("agent_golden: %d cases" % len(cases))


def gen_agent_explicit_gc(pt):
    """The reference's own ValueSimLP with TreeAgent.remove_nodes() (agents/agent.py:246-257, a public method) called by the
    driver between moves whenever fewer than `headroom` slots are free: the collection policy the batched engine offers as
    b200_set_gc_headroom / b200_remove_nodes (one batched collection per move instead of one per overflowing expansion)."""
    from agents.ValueSimLP import ValueSimLP
    out = {}
    cases = [dict(M=6000, sims=40, moves=45, seed=77, headroom=2500), dict(M=5000, sims=30, moves=40, seed=9, headroom=100000)]
    for i, cs in enumerate(cases):
        p = "g%d_" % i
        game = pt.Tetris((20, 10), 1, 0, 0)
        game.seed(cs["seed"])
        ag = ValueSimLP(sims=cs["sims"], env=pt.Tetris, env_args=((20, 10), 1, 0, 0), benchmark=False, online=False, min_visit=40)
        ag.max_nodes = cs["M"]
        ag.init_array()
        ag.model.inference = synthetic_inference
        out[p + "start"] = np.array(game.get_record(), np.uint32)
        ag.update_root(game)
        acts, stats, collected = [], [], []
        for mv in range(cs["moves"]):
            a = ag.play()
            acts.append(int(a))
            stats.append(ag.get_stats())
            game.play(a)
            ag.update_root(game)
            if game.end:
                game.reset()
                ag.update_root(game)
            if len(ag.available) < cs["headroom"]:          # the driver's policy; remove_nodes itself is the reference's
                ag.remove_nodes()
                collected.append(mv)
        out[p + "M"], out[p + "sims"], out[p + "headroom"] = cs["M"], cs["sims"], cs["headroom"]
        out[p + "actions"], out[p + "stats"] = np.array(acts, np.int32), np.stack(stats).astype(np.float32)
        out[p + "collected"] = np.array(collected, np.int32)
        for k in ("child", "score", "episode"):
            out[p + k] = ag.arrays[k]
        out[p + "n2o"] = ag.node_to_obs
        for k in ("visit", "value", "variance"):
            out[p + k] = ag.obs_arrays[k]
        out[p + "root"] = ag.root
        out[p + "n_free"] = len(ag.available)
    out["n_cases"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "agent_gc_golden.npz"), **out)
    print("agent_gc_golden: %d cases, collections at moves %s" % (len(cases), [list(out["g%d_collected" % i])[:8] for i in range(len(cases))]))


def gen_agent_modes(pt):
    """The reference's own agents/ValueSim.py (leaf evaluated, check_low with low=1 draws rand()) and agents/Vanilla.py (random
    rollouts via random.randint, check_low with low=5) on the oracle env.  Their random source is redirected to the oracle's
    per-agent xorshift stream without touching a reference file: the process runs with oracle/_ref/librandshim.so LD_PRELOADed
    (the reference's compiled core.cpp calls its rand()), and the module attribute Vanilla.randint is pointed at the same stream."""
    import ctypes
    shim = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "librandshim.so"))
    shim.shim_next.restype = ctypes.c_uint32
    shim.shim_seed.argtypes = [ctypes.c_uint32]
    if ctypes.CDLL(None).rand != shim.rand and "librandshim" not in os.environ.get("LD_PRELOAD", ""):
        raise RuntimeError("run with LD_PRELOAD=oracle/_ref/librandshim.so (gen_golden.py --agent-modes re-executes itself that way)")
    import agents.Vanilla as RV
    from agents.ValueSim import ValueSim
    RV.randint = lambda a, b: a + int(shim.shim_next() % (b - a + 1))        # Vanilla.py:52 randint(0, n_actions - 1)
    out = {}
    cases = [dict(kind="single", M=6000, sims=40, moves=30, seed=123, search_seed=0x1234567),
             dict(kind="vanilla", M=6000, sims=60, moves=30, seed=321, search_seed=0x7654321),
             dict(kind="single", M=1500, sims=30, moves=40, seed=5, search_seed=99)]       # with garbage collection
    for i, cs in enumerate(cases):
        p = "m%d_" % i
        game = pt.Tetris((20, 10), 1, 0, 0)
        game.seed(cs["seed"])
        if cs["kind"] == "single":
            ag = ValueSim(sims=cs["sims"], env=pt.Tetris, env_args=((20, 10), 1, 0, 0), benchmark=False, online=False, min_visit=40)
            ag.model.inference = synthetic_inference
        else:
            ag = RV.Vanilla(sims=cs["sims"], env=pt.Tetris, env_args=((20, 10), 1, 0, 0), benchmark=False, online=False, min_visit=40)
        ag.max_nodes = cs["M"]
        ag.init_array()
        shim.shim_seed(cs["search_seed"])
        out[p + "start"] = np.array(game.get_record(), np.uint32)
        ag.update_root(game)
        acts, stats = [], []
        for mv in range(cs["moves"]):
            a = ag.play()
            acts.append(int(a))
            stats.append(ag.get_stats())
            game.play(a)
            ag.update_root(game)
            if game.end:
                game.reset()
                ag.update_root(game)
        out[p + "mode"] = 1 if cs["kind"] == "single" else 2
        out[p + "M"], out[p + "sims"], out[p + "search_seed"] = cs["M"], cs["sims"], cs["search_seed"]
        out[p + "actions"], out[p + "stats"] = np.array(acts, np.int32), np.stack(stats).astype(np.float32)
        for k in ("child", "score", "episode"):
            out[p + k] = ag.arrays[k]
        out[p + "n2o"] = ag.node_to_obs
        for k in ("visit", "value", "variance"):
            out[p + k] = ag.obs_arrays[k]
        out[p + "root"] = ag.root
    out["n_cases"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "agent_modes_golden.npz"), **out)
    print("agent_modes_golden: %d cases (ValueSim.py, Vanilla.py, ValueSim.py with collections)" % len(cases))


def gen_agent_cpp(pt):
    """The reference's own C++ agent twin (agents/cppmodule/agent.cpp compiled unchanged -> oracle/_ref/agent*.so): MCTSAgent with
    leaf parallelisation and the synthetic evaluator as its Python callback.  Its LP backup differs from the Python path in two
    places (SURVEY N1: `end` read from the observation, agent.cpp:538; variance averaged without gamma^2, agent.cpp:558) — the
    flags lp_end_from_obs / lp_var_gamma2 of oracle and engine.  The module only exposes play(), so the pinned quantities are
    the action and the game record after every move (arena large enough that its remove_nodes, defective per SURVEY N2, never runs)."""
    agent_mod = O.load_ref_module("agent")

    def evaluator(obs):                                   # agent.cpp:430-434: char[k,1,20,10] -> [values, variances]
        v, var = synthetic_inference(np.asarray(obs).astype(np.int8))
        return [v[:, 0].tolist(), var[:, 0].tolist()]

    out = {}
    cases = [dict(sims=60, moves=50, seed=123), dict(sims=25, moves=120, seed=4242)]
    for i, cs in enumerate(cases):
        p = "c%d_" % i
        game = pt.Tetris((20, 10), 1, 0, 0)
        game.seed(cs["seed"])
        ag = agent_mod.MCTSAgent(cs["sims"], 100000, True, 0.999, True, evaluator, 0, True)   # sims, max_nodes, projection, gamma, benchmark, eval, type, LP
        out[p + "start"] = np.array(game.get_record(), np.uint32)
        ag.update_root(game)
        acts, recs = [], []
        for mv in range(cs["moves"]):
            a = ag.play()
            acts.append(int(a))
            game.play(a)
            recs.append(np.array(game.get_record(), np.uint32))
            ag.update_root(game)
            if game.end:
                game.reset()
                ag.update_root(game)
        out[p + "sims"] = cs["sims"]
        out[p + "actions"], out[p + "records"] = np.array(acts, np.int32), np.stack(recs)
    out["n_cases"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "agent_cpp_golden.npz"), **out)
    print("agent_cpp_golden: %d cases, %s moves" % (len(cases), [c["moves"] for c in cases]))




ONLINE_CASES = {0: dict(memory_size=400, ept=2, growth=150, sims=12, M=2500, moves=420, seed=31, min_visit=3),
                1: dict(memory_size=300, ept=3, growth=150, sims=12, M=2500, moves=420, seed=32, min_visit=3),
                2: dict(memory_size=300, ept=3, growth=150, sims=12, M=2500, moves=420, seed=33, min_visit=3),
                3: dict(memory_size=400, ept=2, growth=90, sims=12, M=2500, moves=420, seed=34, min_visit=3)}


def gen_agent_cpp_online(pt, policy):
    """One accumulation policy of the reference's own OnlineMCTSAgent (agents/cppmodule/agent.cpp:571-820 compiled unchanged, online=True,
    benchmark=False): every train(m_state, m_value, m_variance, m_visit, memory_index) call (agent.cpp:698) is recorded — when it happens
    (move index) and the memory it is handed — together with the actions played.  A fresh process per policy: the reference's random source
    (std::mt19937 mt(123), agent.cpp:29) and random_trimming's IntSampler (a function-static, agent.cpp:752) are process-global."""
    agent_mod = O.load_ref_module("agent")
    cs = ONLINE_CASES[policy]

    def evaluator(obs):                                   # agent.cpp:430-434
        v, var = synthetic_inference(np.asarray(obs).astype(np.int8))
        return [v[:, 0].tolist(), var[:, 0].tolist()]

    calls, move_now = [], [0]

    def train(state, value, variance, visit, n):          # agent.cpp:698
        calls.append((move_now[0], np.array(state[:n, 0], np.int8), np.array(value[:n, 0], np.float32), np.array(variance[:n, 0], np.float32),
                      np.array(visit[:n, 0], np.float32)))

    game = pt.Tetris((20, 10), 1, 0, 0)
    game.seed(cs["seed"])
    ag = agent_mod.OnlineMCTSAgent(sims=cs["sims"], max_nodes=cs["M"], online=True, accumulation_policy=policy, memory_size=cs["memory_size"],
                                   episodes_per_train=cs["ept"], memory_growth_rate=cs["growth"], min_visit=cs["min_visit"], projection=True,
                                   gamma=0.999, benchmark=False, evaluator=evaluator, evaluation_type=0, train=train, LP=True)
    out = {"start": np.array(game.get_record(), np.uint32)}
    ag.update_root(game)
    acts = []
    for mv in range(cs["moves"]):
        move_now[0] = mv
        a = ag.play()
        acts.append(int(a))
        game.play(a)
        ag.update_root(game)
        if game.end:
            game.reset()
            ag.update_root(game)
    out["actions"] = np.array(acts, np.int32)
    # only the actions are kept: the memories handed to train() depend on a defect of TreeAgent::update_available (agent.cpp:300-301, stale
    # `occupied` entries in std::unordered_set order; oracle/agent_probe.cpp) and are pinned through the probe instead (gen_replay_policy)
    for k, v in cs.items():
        out["cfg_" + k] = v
    np.savez_compressed(os.path.join(HERE, "_online_p%d.npz" % policy), **out)
    print("agent_online policy %d: %d train calls at moves %s, rows %s" % (policy, len(calls), [c[0] for c in calls][:12], [len(c[2]) for c in calls][:12]))


def merge_online():
    out = {}
    for p in range(4):
        f = os.path.join(HERE, "_online_p%d.npz" % p)
        z = np.load(f)
        for k in z.files:
            out["p%d_%s" % (p, k)] = z[k]
        os.remove(f)
    np.savez_compressed(os.path.join(HERE, "agent_online_golden.npz"), **out)



PROBE_CASES = {0: dict(memory_size=300, ept=3, growth=100, min_visit=3), 1: dict(memory_size=300, ept=3, growth=100, min_visit=3),
               2: dict(memory_size=300, ept=3, growth=100, min_visit=3), 3: dict(memory_size=300, ept=3, growth=70, min_visit=3)}


def gen_replay_policy(policy):
    """replay_policy_golden: the reference's own OnlineMCTSAgent::remove_nodes (store_nodes incl. the policy-0 random drop, accumulation policies
    0-3, weighted_trimming, random_trimming, the train callback; agent.cpp:619-819, compiled UNCHANGED by inclusion into oracle/_ref/agent_probe)
    driven with scripted collections: each one frees a seeded list of observations (index, visit, value, variance, end, state) at a given
    episode count.  Recorded: memory_index / n_trains after every collection and the memory handed to every train() call.  One process per policy
    (std::mt19937 mt(123) and random_trimming's IntSampler are process-global in the reference)."""
    probe = O.load_ref_module("agent_probe")
    cs = PROBE_CASES[policy]
    M = 4000
    calls = []

    def train(state, value, variance, visit, n):
        calls.append((np.array(state[:n, 0], np.int8), np.array(value[:n, 0], np.float32), np.array(variance[:n, 0], np.float32), np.array(visit[:n, 0], np.float32)))

    pr = probe.Probe(policy, cs["memory_size"], cs["ept"], cs["growth"], cs["min_visit"], M, train)
    rng = np.random.default_rng(100 + policy)
    out = {"n_collections": 36}
    episode = 0
    for c in range(36):
        k = int(rng.integers(20, 150))
        idx = np.sort(rng.choice(np.arange(1, M), k, replace=False)).astype(np.int32)
        visit = rng.integers(1, 220, k).astype(np.int32)
        visit[rng.random(k) < 0.3] = rng.integers(1, 12, int((rng.random(k) < 0.3).sum()) or 1)[0]
        value = rng.uniform(0, 90, k).astype(np.float32)
        variance = rng.uniform(0.05, 500, k).astype(np.float32)
        end = (rng.random(k) < 0.08).astype(np.int32)
        states = ((idx[:, None].astype(np.int64) * 31 + np.arange(200)[None, :] * 17 + c) % 3 - 1).astype(np.int8)   # a formula, so the fixture stays small
        if c % 3 == 2:
            episode += 1
        n_before = len(calls)
        pr.collect(idx.tolist(), visit.tolist(), value.tolist(), variance.tolist(), end.tolist(), states, episode)
        p = "c%d_" % c
        out[p + "idx"], out[p + "visit"], out[p + "value"], out[p + "variance"], out[p + "end"], out[p + "states"] = idx, visit, value, variance, end, states
        out[p + "episode"], out[p + "memory_index"], out[p + "n_trains"], out[p + "trained"] = episode, pr.memory_index(), pr.n_trains(), len(calls) - n_before
    out["n_calls"] = len(calls)
    for i, cl in enumerate(calls):
        out["t%d_state" % i], out["t%d_value" % i], out["t%d_variance" % i], out["t%d_visit" % i] = cl
    for kk, v in cs.items():
        out["cfg_" + kk] = v
    np.savez_compressed(os.path.join(HERE, "_probe_p%d.npz" % policy), **out)
    print("replay_policy %d: %d train calls, rows %s, memory_index trail %s" % (policy, len(calls), [len(c[1]) for c in calls],
                                                                                 [int(out["c%d_memory_index" % c]) for c in range(36)][:14]))


def merge_probe():
    out = {}
    for p in range(4):
        f = os.path.join(HERE, "_probe_p%d.npz" % p)
        z = np.load(f)
        for k in z.files:
            out["p%d_%s" % (p, k)] = z[k]
        os.remove(f)
    np.savez_compressed(os.path.join(HERE, "replay_policy_golden.npz"), **out)


def legacy_torch_overloads():
    """The reference's training code calls torch-1.x overloads that torch 2.x removed: Tensor.add_(Number alpha, Tensor other) and
    Tensor.add(Number, Tensor) (model/model_vv.py:100, model/yogi.py:71,74), addcmul_(Number, Tensor, Tensor) (yogi.py:78-82),
    addcdiv_(Number, Tensor, Tensor) (yogi.py:88).  To RUN THE REFERENCE FILES UNMODIFIED this generator re-creates exactly those
    signatures on torch.Tensor for the duration of the run (alpha-first forms forwarded to the modern keyword forms; same arithmetic)."""
    import numbers
    import torch
    T = torch.Tensor
    orig = dict(add_=T.add_, add=T.add, addcmul_=T.addcmul_, addcdiv_=T.addcdiv_)

    def add_(self, *a, **k):
        if len(a) == 2 and isinstance(a[0], numbers.Number) and isinstance(a[1], torch.Tensor):
            return orig["add_"](self, a[1], alpha=a[0])
        return orig["add_"](self, *a, **k)

    def add(self, *a, **k):
        if len(a) == 2 and isinstance(a[0], numbers.Number) and isinstance(a[1], torch.Tensor):
            return orig["add"](self, a[1], alpha=a[0])
        return orig["add"](self, *a, **k)

    def addcmul_(self, *a, **k):
        if len(a) == 3 and isinstance(a[0], numbers.Number):
            return orig["addcmul_"](self, a[1], a[2], value=a[0])
        return orig["addcmul_"](self, *a, **k)

    def addcdiv_(self, *a, **k):
        if len(a) == 3 and isinstance(a[0], numbers.Number):
            return orig["addcdiv_"](self, a[1], a[2], value=a[0])
        return orig["addcdiv_"](self, *a, **k)

    T.add_, T.add, T.addcmul_, T.addcdiv_ = add_, add, addcmul_, addcdiv_
    return orig


def gen_train():
    """train_golden.npz: the reference's own Model_VV (model/model_vv.py:104-231, torch CPU, Yogi model/yogi.py) taking optimiser steps on a
    seeded batch — Model.train(batch, weighted=...) (model/model.py:95-119) called exactly as Model.train_data does (:207-209).
    Recorded: loss / loss_std / gradient norm of every step, the gradients of the first step, the weights and the optimiser state after
    the last step (large tensors strided), Model.compute_loss on a validation chunk, and a clipped-gradient step."""
    import torch
    from model.model_vv import Model_VV
    torch.set_num_threads(1)
    legacy_torch_overloads()
    rng = np.random.default_rng(11)
    n = 96
    g = O.Game(seed=9)
    states = []
    while len(states) < n:                                    # positions of real (random-play) games: {0, 1, -1} as agents/agent.py:122 stores them
        if g.end:
            g.reset()
        g.play(int(rng.integers(0, 7)))
        states.append(g.state())
    states = np.stack(states).astype(np.int8)
    value = rng.uniform(0, 60, (n, 1)).astype(np.float32)
    variance = rng.uniform(0.0, 400, (n, 1)).astype(np.float32)
    variance[:6] = 0.01                                       # below variance_bound: clamped to 0.1 (model_vv.py:140)
    visit = rng.integers(25, 400, (n, 1)).astype(np.float32)
    weight = (visit / visit.mean()).astype(np.float32)        # model/model.py:186-187
    out = dict(states=states, value=value, variance=variance, weight=weight, seed=0)
    names = ["head.conv1.weight", "head.conv1.bias", "head.conv2.weight", "head.conv2.bias", "head.conv3.weight", "head.conv3.bias",
             "head.fc1.weight", "head.fc1.bias", "head.fc_out.weight", "head.fc_out.bias"]

    def fresh():
        m = Model_VV(use_cuda=False)
        sd = {k: torch.from_numpy(v.copy()) for k, v in O.weights_to_state_dict(O.seeded_weights(0)).items()}
        m.model.load_state_dict(sd)
        m.model.out_ubound = torch.tensor([float(value.max()), float(variance.max())])     # Model_VV.train_data, model_vv.py:227-231
        m.training(True)
        return m

    def flat(m, what):
        params = dict(m.model.named_parameters())
        if what == "w":
            return np.concatenate([params[k].detach().numpy().ravel() for k in names]).astype(np.float32)
        if what == "g":
            return np.concatenate([params[k].grad.detach().numpy().ravel() for k in names]).astype(np.float32)
        st = m.optimizer.state
        return np.concatenate([st[params[k]][what].detach().numpy().ravel() for k in names]).astype(np.float32)

    batch = lambda: [states[:, None, :, :].astype(np.float32), value.copy(), variance.copy(), weight.copy()]   # noqa: E731
    out["ubound"] = np.array([value.max(), variance.max()], np.float32)
    for tag, weighted, clip, steps in (("w", True, 0.0, 3), ("u", False, 0.0, 1), ("c", True, 0.5, 1)):
        m = fresh()
        rec = []
        for it in range(steps):
            r = m.train(batch(), grad_clip=clip, weighted=weighted)
            rec.append([r["loss"], r["loss_std"], r["grad_norm"]])
            if it == 0:
                out[tag + "_grad0"] = flat(m, "g")            # p.grad after the first backward (after clipping when clip > 0)
        out[tag + "_steps"] = np.array(rec, np.float64)
        out[tag + "_weights"] = flat(m, "w")
        if tag == "w":
            out[tag + "_exp_avg"] = flat(m, "exp_avg")
            out[tag + "_exp_avg_sq"] = flat(m, "exp_avg_sq")
            m.training(False)
            val = m.compute_loss([b[:40] for b in batch()], weighted=True, chunksize=16)     # model/model.py:52-83
            out["w_val"] = np.array([val["loss"], val["loss_std"]], np.float64)
            v, var = m.inference(states[:8, None, :, :])
            out["w_pred"] = np.concatenate([v, var], axis=1).astype(np.float32)
    # keep the fixture small: fc1.weight (458752 values) strided, everything else in full
    lo, hi = 18816, 18816 + 458752
    keep = np.ones(478338, bool)
    keep[lo:hi] = False
    keep[lo:hi:97] = True
    out["keep_index"] = np.nonzero(keep)[0].astype(np.int32)
    for k in list(out):
        if isinstance(out[k], np.ndarray) and out[k].shape == (478338,):
            out[k] = out[k][keep]
    np.savez_compressed(os.path.join(HERE, "train_golden.npz"), **out)
    print("train_golden: %d samples; steps (loss, std, gnorm):\n%s" % (n, out["w_steps"]))


def gen_dist():
    """Outputs of the reference's own numba cores (agents/core_distributional.py) on seeded inputs."""
    import agents.core_distributional as R
    from arena_gen import make_dist_arena
    out = {}
    rng = np.random.default_rng(5)
    n = 10
    for i in range(n):
        p = "d%d_" % i
        a = make_dist_arena(i, M=256, bins=50, max_depth=5)
        dist = rng.random(50).astype(np.float32) ** 3
        dist /= dist.sum()
        x = float(rng.uniform(0, 4000))
        out[p + "dist"], out[p + "x"] = dist, x
        out[p + "shift"] = R.shift_distribution(dist, x, 0.0, 5000.0)
        m, v = R.mean_variance(dist, 0.0, 5000.0)
        out[p + "mv"] = np.array([m, v])
        for k in ("child", "node_stats", "node_dist"):
            out[p + k] = a[k]
        # select_trace_distributional itself cannot run upstream: numba 0.65 fails to compile it, and un-jitted it raises in
        # check_low(_child_nodes, node_stats, n) because `count[i] < n` is evaluated on a whole node_stats ROW
        # (core_distributional.py:101 -> agents/core.py:464).  The per-level decision is therefore pinned through the
        # reference's own jitted policy_dist (core_distributional.py:66-79), driven level by level here.
        tr, idx = [], 1
        while True:
            tr.append(idx)
            cn = sorted(set(int(c) for c in a["child"][idx] if c != 0))
            if not cn:
                break
            idx = int(R.policy_dist(np.array(cn, np.int32), a["node_stats"], a["node_dist"], float(a["node_stats"][idx][2]), 0.0, 5000.0))
        out[p + "trace"] = np.asarray(tr, np.int32)
        ns, nd = a["node_stats"].copy(), a["node_dist"].copy()
        r = float(a["node_stats"][tr[-1], 2] + rng.uniform(0, 300))
        R.backup_trace_distributional(np.asarray(tr, np.int32), ns, nd, r, dist, 0.0, 5000.0)
        out[p + "r"], out[p + "bk_stats"] = r, ns
        if i < n - 2:
            out[p + "bk_dist"] = nd
        else:   # keeps the file under 1 MB: only the rows the backup changed (the rest equal node_dist), see arena_gen.golden_bk_dist
            rows = np.nonzero((nd != a["node_dist"]).any(axis=1))[0].astype(np.int32)
            out[p + "bk_rows"], out[p + "bk_dist_rows"] = rows, nd[rows]
    out["n_cases"] = n
    np.savez_compressed(os.path.join(HERE, "dist_golden.npz"), **out)
    print("dist_golden: %d cases" % n)


if __name__ == "__main__":
    O.build(ref=True)
    shim_path = os.path.join(ROOT, "oracle", "_ref", "librandshim.so")
    if "--agent-modes" in sys.argv and "librandshim" not in os.environ.get("LD_PRELOAD", ""):
        # the ValueSim.py / Vanilla.py goldens need the reference's rand() on the oracle's stream: re-execute with the shim preloaded
        # (only this generator: the other goldens are produced with the process's ordinary libc)
        os.environ["LD_PRELOAD"] = shim_path + (":" + os.environ["LD_PRELOAD"] if os.environ.get("LD_PRELOAD") else "")
        os.execv(sys.executable, [sys.executable] + sys.argv)
    pt, core = O.mount_reference()
    if "--dist" in sys.argv:
        gen_dist()
    elif "--train" in sys.argv:
        gen_train()
    elif "--agent-online" in sys.argv:
        gen_agent_cpp_online(pt, int(sys.argv[sys.argv.index("--agent-online") + 1]))
    elif "--replay-policy" in sys.argv:
        gen_replay_policy(int(sys.argv[sys.argv.index("--replay-policy") + 1]))
    elif "--replay-policy-all" in sys.argv:
        import subprocess
        for pol in range(4):
            subprocess.run([sys.executable, os.path.abspath(__file__), "--replay-policy", str(pol)], check=True, stderr=subprocess.DEVNULL)
        merge_probe()
    elif "--agent-online-all" in sys.argv:
        import subprocess
        for pol in range(4):
            subprocess.run([sys.executable, os.path.abspath(__file__), "--agent-online", str(pol)], check=True, stderr=subprocess.DEVNULL)
        merge_online()
    elif "--agent-gc" in sys.argv:
        gen_agent_explicit_gc(pt)
    elif "--agent-modes" in sys.argv:
        gen_agent_modes(pt)
    elif "--agent-cpp" in sys.argv:
        gen_agent_cpp(pt)
    elif "--core-live" in sys.argv:
        gen_core_live(core)
    else:
        gen_core(core)
        gen_core_live(core)
        gen_valuenet()
        gen_agent(pt)
        gen_agent_explicit_gc(pt)
        gen_agent_cpp(pt)
        gen_dist()
        gen_train()
        import subprocess
        subprocess.run([sys.executable, os.path.abspath(__file__), "--agent-online-all"], check=True)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--replay-policy-all"], check=True)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--agent-modes"], check=True)
