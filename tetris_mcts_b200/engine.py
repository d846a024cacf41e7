"""BatchedEngine — N independent game trees searched in lock-step on one B200.

Host-side mirror of the reference's TreeAgent loop (agents/agent.py:147-151 play(), :296-301 update_root(),
:153-185 compute_stats/get_action) for a batch of games; the compute is entirely in libb200_tetris_mcts.so."""
import ctypes as C
import os

import numpy as np

from . import _lib as L


PATH_CACHE_DEFAULT = "1"   # measured on B200 (profiles/exp_path_cache_r2*.txt): 16384 games x 500 sims, move 0.362 -> 0.340 s; results identical (tests)


class BatchedEngine:
    def __init__(self, n_games, max_nodes=8192, mode="lp", gamma=None, low=None, eval_kind="net", weights=None,
                 env_args=((20, 10), 1, 0, 0), seed=123, device=0, lp_end_from_obs=False, lp_var_gamma2=True,
                 stale_pop=True, rollout_variance=1e3, trace_max=512, overflow_reset=False, dist_bins=50, dist_vmin=0.0, dist_vmax=5000.0,
                 dist_weights=None, path_cache=None):
        mode_id = {"lp": L.MODE_LP, "single": L.MODE_SINGLE, "vanilla": L.MODE_VANILLA, "dist": L.MODE_DIST}[mode] if isinstance(mode, str) else int(mode)
        eval_id = {"synthetic": L.EVAL_SYNTHETIC, "net": L.EVAL_NET, "net_tc": L.EVAL_NET_TC}[eval_kind] if isinstance(eval_kind, str) else int(eval_kind)
        if tuple(env_args[0]) != (20, 10):
            raise ValueError("only 20x10 boards (SPEC_PYTETRIS.md §1)")
        cfg = L.Config()
        cfg.n_games, cfg.max_nodes, cfg.mode = int(n_games), int(max_nodes), mode_id
        # reference defaults: ValueSim.py:14 gamma=0.999, ValueSimLP.py:27 low=1; Vanilla.py:9 gamma=0.99, :27 low=5
        cfg.gamma = float(gamma if gamma is not None else (0.99 if mode_id == L.MODE_VANILLA else 0.999))
        # distributional cores: select_trace_distributional(..., low=5) (agents/core_distributional.py:83)
        cfg.low = int(low if low is not None else (5 if mode_id in (L.MODE_VANILLA, L.MODE_DIST) else 1))
        cfg.dist_bins, cfg.dist_vmin, cfg.dist_vmax = int(dist_bins), float(dist_vmin), float(dist_vmax)
        cfg.lp_end_from_obs, cfg.lp_var_gamma2, cfg.stale_pop = int(lp_end_from_obs), int(lp_var_gamma2), int(stale_pop)
        cfg.eval_kind, cfg.trace_max, cfg.overflow_reset = eval_id, int(trace_max), int(overflow_reset)
        cfg.actions_per_drop, cfg.scoring, cfg.randomizer = int(env_args[1]), int(env_args[2]), int(env_args[3])
        cfg.device, cfg.seed, cfg.rollout_variance = int(device), int(seed) & 0xffffffff, float(rollout_variance)
        self.cfg = cfg
        self.n_games, self.max_nodes, self.mode, self.eval_kind = int(n_games), int(max_nodes), mode_id, eval_id
        self.h = L.P()
        self.path_cache = False
        L.check(L.lib().b200_engine_create(C.byref(cfg), C.byref(self.h)))
        if weights is not None:
            self.load_weights(weights)
        if dist_weights is not None:
            self.load_dist_weights(dist_weights, dist_bins)
        # path cache (b200_set_path_cache): None = the default (environment B200_PATH_CACHE, else PATH_CACHE_DEFAULT) wherever it applies
        # (LP mode, max_nodes <= 65536); True / False = explicit (True raises where it does not apply)
        if path_cache is None:
            want = os.environ.get("B200_PATH_CACHE", PATH_CACHE_DEFAULT) not in ("0", "")
            if want and mode_id == L.MODE_LP and int(max_nodes) <= 65536:
                self.set_path_cache(True)
        elif path_cache:
            self.set_path_cache(True)

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "h", None):
            L.lib().b200_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ weights (model/model.py:163-174 Model.load)
    def load_weights(self, weights):
        w = np.ascontiguousarray(weights, np.float32).ravel()
        if w.size != L.N_WEIGHTS:
            raise ValueError("expected %d floats (state_dict order), got %d" % (L.N_WEIGHTS, w.size))
        L.check(L.lib().b200_load_weights(self.h, L.ptr(w)))

    def load_dist_weights(self, weights, atoms=50):
        """model/model_distributional.py Net state_dict tensors concatenated (seq.conv1 ... seq.fc_v)."""
        w = np.ascontiguousarray(weights, np.float32).ravel()
        need = 512 + 32 + 16384 + 32 + 128 * 2048 + 128 + atoms * 128 + atoms
        if w.size != need:
            raise ValueError("expected %d floats, got %d" % (need, w.size))
        L.check(L.lib().b200_load_dist_weights(self.h, L.ptr(w), int(atoms)))
        self._atoms = int(atoms)

    def distnet(self, states):
        s = np.ascontiguousarray(states, np.int8).reshape(-1, 200)
        out = np.zeros((len(s), self._atoms), np.float32)
        L.check(L.lib().b200_distnet_forward(self.h, L.ptr(s), len(s), self._atoms, L.ptr(out)))
        return out

    def export_dist(self, game):
        ns = np.zeros((self.max_nodes, 5), np.float32)
        nd = np.zeros((self.max_nodes, int(self.cfg.dist_bins)), np.float32)
        L.check(L.lib().b200_export_dist(self.h, int(game), L.ptr(ns), L.ptr(nd)))
        return ns, nd

    # ------------------------------------------------------------------ games
    def set_games(self, recs):
        recs = np.ascontiguousarray(recs, np.uint32).reshape(self.n_games, L.REC_WORDS)
        L.check(L.lib().b200_set_games(self.h, L.ptr(recs)))

    def get_games(self):
        recs = np.zeros((self.n_games, L.REC_WORDS), np.uint32)
        L.check(L.lib().b200_get_games(self.h, L.ptr(recs)))
        return recs

    def remove_nodes(self, min_free=2**31 - 1):
        """TreeAgent.remove_nodes() (agents/agent.py:246-257) on every game with fewer than min_free free slots, batched."""
        L.check(L.lib().b200_remove_nodes(self.h, int(min_free)))

    def set_gc_headroom(self, min_free):
        """update_root() then collects every game with fewer than min_free free slots (0 = the reference's lazy collection only)."""
        L.check(L.lib().b200_set_gc_headroom(self.h, int(min_free)))

    def set_path_cache(self, on=True):
        """Keep the children's statistics of every trace level next to the trace, so that the next walk of the game (which retraces ~93 % of the
        path) reads one sequential line per level instead of two dependent random accesses.  No effect on results.  LP mode, max_nodes <= 65536."""
        L.check(L.lib().b200_set_path_cache(self.h, int(bool(on))))
        self.path_cache = bool(on)

    def update_root(self, auto_reset=False):
        L.check(L.lib().b200_update_root(self.h, int(auto_reset)))

    def run_sims(self, sims):
        L.check(L.lib().b200_run_sims(self.h, int(sims)))

    def get_stats(self):
        stats = np.zeros((self.n_games, 3, L.N_ACTIONS), np.float32)
        action = np.zeros(self.n_games, np.int32)
        L.check(L.lib().b200_get_stats(self.h, L.ptr(stats), L.ptr(action)))
        return stats, action

    def env_step(self, actions=None):
        a = None if actions is None else np.ascontiguousarray(actions, np.int32)
        L.check(L.lib().b200_env_step(self.h, L.ptr(a)))

    def play_move(self, sims, auto_reset=True, want_stats=True):
        """One move of play.py:118-177 for every game. Returns (actions, stats)."""
        actions = np.zeros(self.n_games, np.int32)
        stats = np.zeros((self.n_games, 3, L.N_ACTIONS), np.float32) if want_stats else None
        L.check(L.lib().b200_play_move(self.h, int(sims), int(auto_reset), L.ptr(actions), L.ptr(stats)))
        return actions, stats

    def finished_games(self):
        """Episodes that ended (and were reset) since the last call: int32[k,4] rows {game, score, line_clears, episode}, sorted by game
        (play.py:161-177: the numbers of its `Episode:` line)."""
        cap = 4 * self.n_games
        out = np.zeros((cap, 4), np.int32)
        cnt = np.zeros(1, np.int32)
        L.check(L.lib().b200_finished_games(self.h, L.ptr(out), cap, L.ptr(cnt)))
        rows = out[:min(int(cnt[0]), cap)]
        return rows[np.lexsort((rows[:, 3], rows[:, 0]))]

    def sync(self):
        L.check(L.lib().b200_sync(self.h))

    # ------------------------------------------------------------------ SURVEY 8(b).5: explicit cudaStream_t
    def set_stream(self, stream):
        """Issue all work of this engine on the caller's CUDA stream: a raw cudaStream_t handle (int), an object with a `cuda_stream`
        attribute (torch.cuda.Stream), or None for a private stream again.  The caller keeps the stream alive."""
        handle = 0 if stream is None else int(getattr(stream, "cuda_stream", stream))
        L.check(L.lib().b200_engine_set_stream(self.h, C.c_void_p(handle)))

    def get_stream(self):
        """The cudaStream_t (int) the engine issues its work on — e.g. torch.cuda.ExternalStream(engine.get_stream())."""
        out = C.c_void_p()
        L.check(L.lib().b200_engine_get_stream(self.h, C.byref(out)))
        return int(out.value or 0)

    def status(self):
        st = np.zeros(self.n_games, np.int32)
        L.check(L.lib().b200_status(self.h, L.ptr(st)))
        return st

    COUNTER_NAMES = ("sims", "expansions", "eval_requests", "gcs", "trace_levels", "rollout_steps", "new_nodes", "tree_resets",
                     "games_finished", "score_sum", "lines_sum", "_11", "max_trace_len", "cached_levels")

    def counters(self):
        c = np.zeros(16, np.uint64)
        L.check(L.lib().b200_counters(self.h, L.ptr(c)))
        return {n: int(c[i]) for i, n in enumerate(self.COUNTER_NAMES) if not n.startswith("_")}

    PHASES = ("select_expand", "conv", "fc", "backup", "rollout", "synthetic", "misc", "gc")

    def timer_start(self):
        L.check(L.lib().b200_timer_start(self.h))

    def timer_stop(self):
        ms = np.zeros(1, np.float32)
        L.check(L.lib().b200_timer_stop(self.h, L.ptr(ms)))
        return float(ms[0])

    def set_timing(self, on=True):
        L.check(L.lib().b200_set_timing(self.h, int(on)))

    def phase_ms(self):
        ms = np.zeros(8, np.float32)
        n = np.zeros(8, np.uint64)
        L.check(L.lib().b200_phase_ms(self.h, L.ptr(ms), L.ptr(n)))
        return {p: (float(ms[i]), int(n[i])) for i, p in enumerate(self.PHASES) if not p.startswith("_")}

    # ------------------------------------------------------------------ parity / introspection
    def export_game(self, game):
        """The arena of one game in the reference's array layout (agents/agent.py:58-88)."""
        M = self.max_nodes
        d = dict(child=np.zeros((M, 7), np.int32), score=np.zeros(M, np.float32), episode=np.zeros(M, np.int32),
                 n2o=np.zeros(M, np.int32), visit=np.zeros(M, np.int32), value=np.zeros(M, np.float32),
                 variance=np.zeros(M, np.float32), obs_end=np.zeros(M, np.uint8),
                 game=np.zeros((M, L.REC_WORDS), np.uint32), obs_key=np.zeros((M, L.KEY_WORDS), np.uint32))
        root = np.zeros(1, np.int32)
        tr = np.zeros(int(self.cfg.trace_max) or 512, np.int32)
        tl = np.zeros(1, np.int32)
        L.check(L.lib().b200_export_game(self.h, int(game), L.ptr(d["child"]), L.ptr(d["score"]), L.ptr(d["episode"]),
                                         L.ptr(d["n2o"]), L.ptr(d["visit"]), L.ptr(d["value"]), L.ptr(d["variance"]),
                                         L.ptr(d["obs_end"]), L.ptr(d["game"]), L.ptr(d["obs_key"]), L.ptr(root),
                                         L.ptr(tr), L.ptr(tl)))
        d["root"] = int(root[0])
        d["last_trace"] = tr[:int(tl[0])].copy()
        return d

    def valuenet(self, states):
        """Model_VV.inference (model/model_vv.py:210-217): states (k,1,20,10) or (k,20,10) in {-1,0,1} -> (v, var)."""
        s = np.ascontiguousarray(states, np.int8).reshape(-1, 200)
        v = np.zeros(len(s), np.float32)
        var = np.zeros(len(s), np.float32)
        L.check(L.lib().b200_valuenet_forward(self.h, L.ptr(s), len(s), L.ptr(v), L.ptr(var)))
        return v, var

    def replay_enable(self, min_visits=25, capacity=500000):
        """ValueSim(online=True) replay memory (agents/ValueSim.py:14-37; min_visits_to_store=25 for ValueSimLP.py:11)."""
        L.check(L.lib().b200_replay_enable(self.h, int(min_visits), int(capacity)))

    def replay_drain_into(self, dev_ptr, capacity):
        cnt = np.zeros(1, np.int32)
        L.check(L.lib().b200_replay_drain_dev(self.h, C.c_void_p(int(dev_ptr)), int(capacity), L.ptr(cnt)))
        return int(cnt[0])

    def replay_policy(self, accumulation_policy, episodes_per_train=25, memory_growth_rate=5000):
        """OnlineMCTSAgent(accumulation_policy=, episodes_per_train=, memory_growth_rate=) (agent.cpp:588-617) on the memory of replay_enable."""
        L.check(L.lib().b200_replay_policy(self.h, int(accumulation_policy), int(episodes_per_train), int(memory_growth_rate)))

    def replay_policy_step(self, current_episode):
        """The decision of OnlineMCTSAgent::remove_nodes after storing (agent.cpp:632-702) -> (train_now, memory_index)."""
        t, m = np.zeros(1, np.int32), np.zeros(1, np.int32)
        L.check(L.lib().b200_replay_policy_step(self.h, int(current_episode), L.ptr(t), L.ptr(m)))
        return bool(t[0]), int(m[0])

    def replay_policy_trained(self, current_episode):
        L.check(L.lib().b200_replay_policy_trained(self.h, int(current_episode)))

    def replay_append(self, rows):
        """rows uint8[n,212] join the memory as the rows of a collection would (in order, until the memory is full)."""
        r = np.ascontiguousarray(rows, np.uint8).reshape(-1, 212)
        L.check(L.lib().b200_replay_append(self.h, L.ptr(r), len(r)))

    def replay_peek_into(self, dev_ptr, n_rows):
        L.check(L.lib().b200_replay_peek_dev(self.h, C.c_void_p(int(dev_ptr)), int(n_rows)))

    def collect_samples_into(self, dev_ptr, capacity, min_visits):
        """ValueSim.store_nodes-style samples (agents/ValueSim.py:122-159) written to a DEVICE buffer of 212-byte rows."""
        cnt = np.zeros(1, np.int32)
        L.check(L.lib().b200_collect_samples_dev(self.h, int(min_visits), C.c_void_p(int(dev_ptr)), int(capacity), L.ptr(cnt)))
        return int(cnt[0])
