#!/usr/bin/env python
"""bench.py — MCTS simulations/second of the per-move simulation loop (select -> step/expand -> value net -> backup)
over N concurrent games, on 1..8 B200 (one process per GPU), next to the reference's CPU path.

  python bench.py --gpus 1 --steps K --warmup W            B200 arm (this repo's CUDA engine through its C-ABI)
  python bench.py --impl reference --steps K --warmup W    reference arm: the reference's own compiled
                                                            agents/cppmodule/agent.cpp (oracle/_ref) on the host cores
A "step" is one move of every game: `sims` simulations per game, then get_action, play, update_root (play.py:118-177).
Workload (BASELINE.json configs[2], the one north_star's target sentence names: >= 16384 concurrent games, ValueSimLP +
value net, 500 sims/move).  `--workload vanilla` selects configs[1] (Vanilla MCTS, 4096 games, 300 sims/move).
Prints ONE JSON line on rank 0."""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONV_FLOP = 82944 + 1769472 + 1032192          # SURVEY §8a a11: conv1 + conv2 + conv3 per board
FC_FLOP = 917504 + 1024                          # fc1 + fc_out per board
NET_FLOP = CONV_FLOP + FC_FLOP                   # 3 803 136
ENV_ARGS = ((20, 10), 1, 0, 0)                   # play.py:75 defaults
BASE_SEED = 123                                  # SURVEY §8d (echoes agent.cpp:23)


TC_ISSUED_FLOP_PER_BOARD = 2 * 128 * 16 * (96 * 36 + 64 * 2)   # k_tc_conv: 2x18 MMAs of 128x96x16 + 2 of 128x64x16 per board
ARENA_BYTES_PER_SLOT = 304


def _ncu_traffic_file():
    for name in ("ncu_traffic_r2b.json", "ncu_traffic_r2.json", "ncu_traffic_r1.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            return p
    return None


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full capture (profiles/)."""
    try:
        return json.load(open(_ncu_traffic_file())).get(kernel, {}).get("dram_bytes")
    except Exception:
        return None


def ncu_traffic_src():
    """Which capture `traffic` comes from and the regime it was taken in (bench window or not)."""
    try:
        p = _ncu_traffic_file()
        return {"file": os.path.relpath(p, ROOT), "regime": json.load(open(p)).get("_regime", "round-1 capture: moves 0-1 at 100-150 sims (NOT the bench window)")}
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, src="fallback")   # B200_PROFILING.md fallback


# ----------------------------------------------------------------------------------------------- clocks sampler
class Clocks:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.p, self.index = [], None, index

    def __enter__(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None
        return self

    def _read(self):
        for line in self.p.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 7:
                self.rows.append(f)

    def __exit__(self, *a):
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == "Active" for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------- reference arm
def ref_agent_moves(workload, sims, max_nodes):
    """Moves a reference agent object may play before it is replaced by a fresh one (same class, same arguments, re-rooted at the
    live game).  Why: the reference's arena cannot survive a long game — once the reachable set fills max_nodes its own
    remove_nodes() frees nothing, agent.cpp:227-231 prints MAX_NODES EXCEEDED and calls available.back() on an empty vector
    (undefined behaviour: the round-1 arm segfaulted there at ~60 moves), and agent.cpp:300-301 doubles `occupied` on the way.
    A simulation creates at most 7 nodes (agent.cpp:201-208) and update_root one, so max_nodes // (7*sims + 1) moves can never
    exhaust the free list: the unmodified reference code then never reaches its overflow path."""
    return max(1, max_nodes // (7 * sims + 1))


def _ref_worker(conn, wid, workload, sims):
    """One single-threaded worker = one play.py-equivalent process (BASELINE.md §3) on the reference's compiled C++ agent."""
    try:
        os.environ["OMP_NUM_THREADS"] = "1"
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import torch
        torch.set_num_threads(1)
        import oracle_py as O
        from random import randint
        pt = O.load_ref_module("pyTetris")
        agent_mod = O.load_ref_module("agent")          # the reference's own agents/cppmodule/agent.cpp, compiled unchanged
        game = pt.Tetris(*ENV_ARGS)
        game.seed(BASE_SEED + wid)
        if workload == "vanilla":                        # agents/VanillaC.py:5-13
            max_nodes = 500000

            def random_playout(g):
                while not g.end:
                    g.play(randint(0, 7))
                return g.score, 1e5

            def make_agent():
                return agent_mod.MCTSAgent(sims, max_nodes, True, 0.99, True, random_playout, 1, False)
        else:                                            # agents/ValueSimC.py:17-42 (LP=True, evaluator = Model_VV.inference)
            from ref_net import RefModel
            max_nodes = 100000
            model = RefModel(O.weights_to_state_dict(O.seeded_weights(0)))

            def make_agent():
                return agent_mod.OnlineMCTSAgent(sims=sims, max_nodes=max_nodes, online=False, accumulation_policy=3, memory_size=1,
                                                 episodes_per_train=25, memory_growth_rate=5000, min_visit=25, projection=True, gamma=0.999,
                                                 benchmark=True, evaluator=model.inference, evaluation_type=0, train=(lambda *a: None), LP=True)
        renew_after = ref_agent_moves(workload, sims, max_nodes)
        agent = make_agent()
        agent.update_root(game)
        age = 0
        conn.send("ready")
        while True:
            msg = conn.recv()
            if msg[0] == "stop":
                break
            done, renewed, t0 = 0, 0, time.perf_counter()
            if msg[0] == "moves":
                budget_moves, budget_s = msg[1], 1e18
            else:
                budget_moves, budget_s = 1 << 30, msg[1]
            while done < budget_moves and time.perf_counter() - t0 < budget_s:
                if age >= renew_after:                   # inside the timed region: constructing the agent is part of the reference's cost
                    agent = make_agent()
                    agent.update_root(game)
                    age, renewed = 0, renewed + 1
                a = agent.play()
                game.play(a)
                agent.update_root(game)
                if game.end:
                    game.reset()
                    agent.update_root(game)
                done += 1
                age += 1
            conn.send((done * sims, time.perf_counter() - t0, renewed))
    except Exception as ex:   # noqa
        try:
            conn.send(("error", repr(ex)))
        except Exception:
            pass


class RefPool:
    """P single-threaded worker processes.  A worker that dies (the reference's C++ can take the whole process down) is
    detected through its pipe / exit code, replaced by a fresh worker, and its unfinished sample counts as zero simulations."""

    def __init__(self, workload, sims, procs=None):
        self.P = procs or os.cpu_count() or 1
        self.workload, self.sims = workload, sims
        self.ctx = mp.get_context("spawn")
        self.conns, self.procs = [None] * self.P, [None] * self.P
        self.restarts, self.renewals = 0, 0
        for w in range(self.P):
            self._spawn(w)
        for w in range(self.P):
            self._wait_ready(w)

    def _spawn(self, w):
        a, b = self.ctx.Pipe()
        p = self.ctx.Process(target=_ref_worker, args=(b, w, self.workload, self.sims), daemon=True)
        p.start()
        b.close()                                        # so that a dead child gives EOF instead of a hang
        self.conns[w], self.procs[w] = a, p

    def _wait_ready(self, w, tries=3):
        for _ in range(tries):
            try:
                r = self.conns[w].recv()
                if r == "ready":
                    return
                raise RuntimeError("reference worker failed: %r" % (r,))
            except (EOFError, OSError):
                self._spawn(w)
        raise RuntimeError("reference worker %d cannot start" % w)

    def _restart(self, w):
        self.restarts += 1
        try:
            self.conns[w].close()
        except Exception:
            pass
        if self.procs[w].is_alive():
            self.procs[w].kill()
        self.procs[w].join(timeout=5)
        self._spawn(w)
        self._wait_ready(w)

    def run(self, kind, amount):
        """Every worker runs `amount` moves (kind == 'moves') or seconds; returns (simulations done, slowest worker's seconds)."""
        from multiprocessing.connection import wait
        pending = {}
        for w in range(self.P):
            try:
                self.conns[w].send((kind, amount))
                pending[self.conns[w]] = w
            except (BrokenPipeError, OSError):
                self._restart(w)
        t0 = time.perf_counter()
        n_tot, t_max = 0, 0.0
        while pending:
            for c in wait(list(pending), timeout=5.0):
                w = pending.pop(c)
                try:
                    r = c.recv()
                except (EOFError, OSError):
                    r = None
                if r is None or r[0] == "error":          # died inside the reference's code: replace it, its sample is lost
                    if r is not None:
                        sys.stderr.write("reference worker %d: %s\n" % (w, r[1]))
                    self._restart(w)
                    t_max = max(t_max, time.perf_counter() - t0)
                    continue
                n_tot += r[0]
                t_max = max(t_max, r[1])
                self.renewals += r[2]
        return n_tot, t_max

    def close(self):
        for c in self.conns:
            try:
                c.send(("stop",))
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=10)
            if p.is_alive():
                p.kill()


REF_ARM_NOTE = ("the reference's own compiled agents/cppmodule/agent.cpp (oracle/_ref, unmodified) driven as agents/ValueSimC.py:17-42 / VanillaC.py:5-13 "
                "do: one game per single-threaded worker process, one worker per host core, torch fp32 CPU value net as the evaluator callback; "
                "env = the oracle restatement of pyTetris (absent upstream).  The agent object is replaced by a fresh one (same arguments, "
                "re-rooted at the live game, construction inside the timed region) every max_nodes // (7*sims+1) moves so that the reference never "
                "reaches its arena-overflow path (agent.cpp:224-231, undefined behaviour); a worker that dies anyway is restarted and its sample lost")


def cpu_baseline(workload, sims, seconds):
    pool = RefPool(workload, sims)
    try:
        pool.run("seconds", min(2.0, seconds / 4))          # warm-up (JIT of the scripted net, caches)
        n, t = pool.run("seconds", seconds)
    finally:
        pool.close()
    return {"value": n / t, "unit": "sims/s", "cores": pool.P, "kind": "reference",
            "sample": "%d single-threaded workers x ~%.0f s of %s at %d sims/move on the reference's compiled agent.cpp + torch fp32 CPU net "
                      "(env = oracle restatement: pyTetris is absent upstream); %d sims total; %d worker restarts"
                      % (pool.P, seconds, workload, sims, n, pool.restarts)}


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    sims = cfg["sims"]
    pool = RefPool(cfg["workload_key"], sims)
    try:
        moves_per_step = args.ref_moves_per_step
        for _ in range(args.warmup):
            pool.run("moves", moves_per_step)
        r0, n0 = pool.restarts, pool.renewals
        tot_n, tot_t = 0, 0.0
        for _ in range(args.steps):
            n, t = pool.run("moves", moves_per_step)
            tot_n += n
            tot_t += t
    finally:
        pool.close()
    value = tot_n / max(tot_t, 1e-9)
    max_nodes = 500000 if cfg["workload_key"] == "vanilla" else 100000
    sample = ("%d workers x %d moves x %d sims per step; agent renewed every %d moves (%d renewals, %d worker restarts in the timed steps)"
              % (pool.P, moves_per_step, sims, ref_agent_moves(cfg["workload_key"], sims, max_nodes), pool.renewals - n0, pool.restarts - r0))
    line = {"impl": "reference", "metric": "mcts_sims_per_sec", "value": value, "unit": "sims/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg["config"],
            "cpu_baseline": {"value": value, "unit": "sims/s", "cores": pool.P, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "reference_arm": REF_ARM_NOTE + "; `config` is the B200 arm's, for the ratio"}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- B200 arm
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, rank, world):
    """--dump-outputs: what the timed path computed in its last step, one float64 DIR/<name>.npy per array (first axis = game),
    so that two builds run with the same arguments can be compared output for output.  game_index.npy holds the game of every
    row: all games, or, when the files would exceed DUMP_LIMIT_BYTES in all, a fixed sample (numpy PCG64 seed 0).  With
    several ranks every rank writes its own shard under a _rank<r> suffix, within its share of the limit."""
    n = len(next(iter(arrays.values())))
    row_bytes = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))
    keep = min(n, (DUMP_LIMIT_BYTES // world - 4096) // row_bytes)          # 4096: room for the .npy headers
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    suffix = "" if world == 1 else "_rank%d" % rank
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "game_index%s.npy" % suffix), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, "%s%s.npy" % (name, suffix)), np.asarray(a)[idx].astype(np.float64))


def run_b200(args, cfg):
    """Three passes over the SAME workload: the search is deterministic given the seeds (SURVEY N3), so every pass builds an
    identical engine from the same seeds, plays the same W warm-up moves and then the same K moves:
      pass 1  `value`: production path (one CUDA graph per simulation step), inputs resident in HBM, CUDA events on the engine stream
      pass 2  per-kernel launch durations (an event pair around every kernel, direct launches) for the roofline figures
      pass 3  `e2e`: the public API with HOST buffers — H2D of the games, D2H of actions / statistics / games every move, plus the
              path's one exchange step (replay rows drained from the device memory k_gc fills -> all-gather over NCCL when N > 1)
    The per-pass counters (simulations, expansions, evaluations, trace levels) must agree, and the line says so (`same_workload`)."""
    import torch
    from tetris_mcts_b200 import distributed as D
    from tetris_mcts_b200 import pyTetris as PT
    from tetris_mcts_b200.engine import BatchedEngine
    from tetris_mcts_b200.model.model_vv import init_weights

    rank, local_rank, world = D.init()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    G, sims, M = cfg["games_per_gpu"], cfg["sims"], cfg["max_nodes"]
    seeds = D.shard_seeds(BASE_SEED, G * world, rank, world)
    recs = PT.new_games(G, ENV_ARGS, seeds)
    dist_w = None
    if cfg["mode"] == "dist":
        from tetris_mcts_b200.agents.DistValueSimOnline import init_dist_weights
        dist_w = init_dist_weights(0, 50)
    weights = init_weights(0) if cfg["mode"] in ("lp", "single") else None

    def fresh_engine():
        e = BatchedEngine(G, max_nodes=M, mode=cfg["mode"], eval_kind=cfg["eval"], weights=weights, dist_weights=dist_w, env_args=ENV_ARGS,
                          seed=BASE_SEED + 7919 * rank, device=local_rank, rollout_variance=1e3, overflow_reset=True,
                          path_cache={"auto": None, "on": True, "off": False}[args.path_cache])
        e.set_games(recs)
        e.set_gc_headroom(cfg["gc_headroom"])
        return e

    WORK_KEYS = ("sims", "expansions", "eval_requests", "trace_levels", "new_nodes", "gcs", "tree_resets")
    # ---- pass 1: device-timed region (inputs resident in HBM, no host buffers)
    eng = fresh_engine()
    eng_path_cache = bool(getattr(eng, "path_cache", False))
    for _ in range(args.warmup):
        eng.play_move(sims, auto_reset=True, want_stats=False)
    eng.sync()
    c0 = eng.counters()
    eng.set_timing(False)                      # zeroes the launch counters
    D.barrier()
    torch.cuda.synchronize()
    with Clocks(local_rank) as clk:
        eng.timer_start()
        for _ in range(args.steps):
            actions, _ = eng.play_move(sims, auto_reset=True, want_stats=False)
        ms = eng.timer_stop()
    torch.cuda.synchronize()
    D.barrier()
    c1 = eng.counters()
    longest_trace = c1.pop("max_trace_len", None)             # not cumulative: the longest trace of the last move
    c0.pop("max_trace_len", None)
    launches = sum(n for _, n in eng.phase_ms().values())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"actions": actions, "games": eng.get_games()}, rank, world)
    ms_max = D.max_over_ranks(ms, dev)
    delta = {k: c1[k] - c0[k] for k in c1}
    tot = D.sum_over_ranks(delta, dev)
    value = tot["sims"] / (ms_max / 1e3)
    eng.close()
    # ---- pass 2: the same K moves with a CUDA event pair around every kernel.  Not part of `value`.
    eng = fresh_engine()
    for _ in range(args.warmup):
        eng.play_move(sims, auto_reset=True, want_stats=False)
    eng.sync()
    eng.set_timing(True)
    p0 = eng.counters()
    eng.timer_start()
    for _ in range(args.steps):
        eng.play_move(sims, auto_reset=True, want_stats=False)
    ms_instr = eng.timer_stop()
    phases = eng.phase_ms()
    eng.set_timing(False)
    p1 = eng.counters()
    p0.pop("max_trace_len", None); p1.pop("max_trace_len", None)
    pdelta = {k: p1[k] - p0[k] for k in p1}
    eng.close()
    # ---- pass 3: end to end through the public API with HOST buffers; the exchange step inside the loop
    eng = fresh_engine()
    cap = args.exchange_rows
    eng.replay_enable(min_visits=25, capacity=4 * cap)            # ValueSimLP.py:11 min_visits_to_store=25; filled by k_gc (ValueSim.py:101-159)
    block = torch.empty((cap, D.SAMPLE_BYTES), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()                                       # the buffer is handed to the engine's own stream (no cross-stream race)
    pin_recs = torch.empty((G, 20), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
    pin_recs[:] = recs
    gather_ms, rows_seen = [], 0

    def e2e_step(timed):
        nonlocal rows_seen
        eng.set_games(pin_recs)                                   # H2D G*80 B + update_root
        actions, stats = eng.play_move(sims, auto_reset=True)     # D2H G*(4+84) B
        pin_recs[:] = eng.get_games()                             # D2H G*80 B
        n_local = eng.replay_drain_into(block.data_ptr(), cap)    # device -> device, rows stored by this move's collections
        tg = time.perf_counter()
        rows, counts = D.allgather_samples(block, n_local)
        torch.cuda.synchronize()                                  # the block is rewritten by the engine's stream next move
        if timed:
            gather_ms.append((time.perf_counter() - tg) * 1e3)
            rows_seen += int(rows.shape[0])

    for _ in range(args.warmup):
        e2e_step(False)
    eng.sync()
    e0 = eng.counters()
    D.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step(True)
    eng.sync()
    torch.cuda.synchronize()
    e2e_s = D.max_over_ranks(time.perf_counter() - t0, dev)
    D.barrier()
    e1 = eng.counters()
    e0.pop("max_trace_len", None); e1.pop("max_trace_len", None)
    edelta = {k: e1[k] - e0[k] for k in e1}
    e2e_sims = D.sum_over_ranks({"sims": edelta["sims"]}, dev)["sims"]
    eng.close()
    same = all(delta[k] == pdelta[k] == edelta[k] for k in WORK_KEYS)
    gather_ms_max = [D.max_over_ranks(x, dev) for x in gather_ms]
    rows_tot = D.sum_over_ranks({"r": rows_seen}, dev)["r"] / max(world, 1)       # every rank sees all rows after the gather
    traj = {"rows_per_step": rows_tot / max(args.steps, 1), "block_bytes_per_rank": cap * D.SAMPLE_BYTES,
            "ms_median": statistics.median(gather_ms_max) if gather_ms_max else None, "ms_max": max(gather_ms_max) if gather_ms_max else None,
            "iterations": len(gather_ms_max), "backend": "nccl" if world > 1 else "none (1 rank: device-to-device drain only)",
            "source": "b200_replay_drain_dev (rows k_gc stored from the observations this move's collections freed), inside the e2e loop"}
    peaks = measured_peaks()
    out = None
    if rank == 0:
        steps = max(args.steps, 1)
        roof, roof_tree = None, None
        D_mean = pdelta["trace_levels"] / max(pdelta["sims"], 1)
        sel_ms, sel_n = phases["select_expand"]
        bk_ms, bk_n = phases["backup"]
        tree_bytes = pdelta["sims"] * (200.0 * D_mean - 140.0) + pdelta["expansions"] * 1100.0       # SURVEY §8d
        tree_s = (sel_ms + bk_ms) / 1e3
        if tree_s > 0:
            ach = tree_bytes / tree_s / 1e9
            tr_s, tr_b = ncu_traffic("k_select_expand"), ncu_traffic("k_backup")
            roof_tree = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                         "traffic": (tr_s + tr_b) if tr_s and tr_b else None, "traffic_src": ncu_traffic_src(),
                         "algorithmic_bytes_per_launch_pair": tree_bytes / max(sel_n, 1),
                         "kernels": "k_select_expand + k_backup", "mean_trace_len": D_mean, "ms_per_launch_pair": (sel_ms + bk_ms) / max(sel_n, 1),
                         "peak_src": peaks["src"]}
            # The walk is a chain of RANDOM accesses, so the streaming-copy peak is not its ceiling.  scripts/probe/mem_probe.cu measured what this
            # memory system delivers for independent random 64-byte bursts that miss L2 (profiles/mem_probe_r2.txt): 40 G bursts/s (2.6 TB/s) at
            # 1 GB, 31-36 G/s at 8 GB — and 6-10 G/s over a 128 GB footprint (2 MB pages: TLB reach).  The kernels' own DRAM traffic (ncu, same
            # regime) divided by 64 B and by the measured launch time is their burst rate against that ceiling.
            if tr_s and tr_b:
                cap = 40.0e9
                roof_tree["random_access"] = {"ceiling_gbursts_per_s": cap / 1e9, "ceiling_src": "profiles/mem_probe_r2.txt: random 64-byte bursts, 1 GB footprint, 32-64 warps/SM",
                                              "k_select_expand_gbursts_per_s": tr_s / 64.0 / (sel_ms / max(sel_n, 1) / 1e3) / 1e9,
                                              "k_backup_gbursts_per_s": tr_b / 64.0 / (bk_ms / max(bk_n, 1) / 1e3) / 1e9,
                                              "frac_select": tr_s / 64.0 / (sel_ms / max(sel_n, 1) / 1e3) / cap,
                                              "frac_backup": tr_b / 64.0 / (bk_ms / max(bk_n, 1) / 1e3) / cap,
                                              "note": "DRAM bytes of the ncu capture (traffic_src) / 64 B / this run's launch time.  With the path cache on most of "
                                                      "k_select_expand's reads are sequential lines (config.path_cache), so its figure mixes streaming and random "
                                                      "bursts; k_backup's trace records are sequential too (a ratio above 1 is not a contradiction)"}
        if cfg["mode"] == "dist":
            conv_ms, conv_n = phases["conv"]
            flop = 19 * 7 * 32 * 16 * 2 + 16 * 4 * 32 * 512 * 2   # conv1 (19x7 pixels) + conv2 (16x4) on the 22x10 input of model_distributional.py:27
            ach = pdelta["eval_requests"] * flop / max(conv_ms / 1e3, 1e-9) / 1e12
            fc_ms, fc_n = phases["fc"]
            roof = {"bound": "tensor", "achieved": ach, "peak": peaks["tensor"], "unit": "TFLOP/s", "frac": ach / peaks["tensor"], "traffic": None,
                    "kernel": "k_tdc_conv" if cfg["eval"] == "net_tc" else "k_dn_conv", "ms_per_launch": conv_ms / max(conv_n, 1),
                    "share_of_step": conv_ms / ms_instr, "peak_src": peaks["src"] + " bf16 dense, sustained",
                    "fc_kernel_tflops": pdelta["eval_requests"] * 2 * 2048 * 128 / (fc_ms / 1e3) / 1e12 if fc_ms > 0 else None,
                    "note": "achieved counts ALGORITHMIC conv FLOPs (2 233 344 per board).  eval=net_tc: tcgen05 kind::f16 with the fp32 operands split into two "
                            "scaled fp16 terms (k_tdc_conv / k_tdc_fc, csrc/distnet_tc.cuh); eval=net: fp32 CUDA cores (k_dn_conv / k_dn_fc)"}
        elif cfg["mode"] != "vanilla":
            conv_ms, conv_n = phases["conv"]
            fc_ms, fc_n = phases["fc"]
            boards = pdelta["eval_requests"]
            if conv_ms > 0 and conv_n > 0:
                ach = boards * CONV_FLOP / (conv_ms / 1e3) / 1e12
                kname = "k_vn_conv" if cfg["eval"] == "net" else "k_tc_conv"
                roof = {"bound": "tensor", "achieved": ach, "peak": peaks["tensor"], "unit": "TFLOP/s", "frac": ach / peaks["tensor"],
                        "traffic": ncu_traffic(kname), "traffic_src": ncu_traffic_src(), "kernel": kname,
                        "mma_flops_issued_per_launch": boards * TC_ISSUED_FLOP_PER_BOARD / conv_n, "ms_per_launch": conv_ms / conv_n,
                        "flops_per_launch": boards * CONV_FLOP / conv_n, "boards_per_launch": boards / conv_n,
                        "fc_kernel_tflops": boards * FC_FLOP / (fc_ms / 1e3) / 1e12 if fc_ms > 0 else None,
                        "share_of_step": conv_ms / ms_instr, "peak_src": peaks["src"] + " bf16 dense, sustained",
                        "note": "achieved counts ALGORITHMIC conv FLOPs (SURVEY 8d: 2 884 608 per board).  fp32-faithful arithmetic (north_star 1e-5): "
                                "eval=net is CUDA-core fp32 FMA; eval=net_tc is tcgen05 kind::f16 with every fp32 operand split into two scaled fp16 terms "
                                "(3 products per algorithmic product; M=128 pixel tiles carry halo rows), so the tensor pipe executes "
                                "mma_flops_issued_per_launch.  scripts/probe/mma_probe.cu measures SS-mode tcgen05.mma at (A+B operand bytes)/128 B/clk with a "
                                "44.7 clk floor: these small-N MMAs are shared-memory operand-fetch bound, not tensor-rate bound; the bf16 peak is the "
                                "driver-measured denominator, not this kernel's ceiling"}
        else:
            ro_ms, ro_n = phases["rollout"]
            roof = {"bound": "hbm", "achieved": 0.0, "peak": peaks["hbm"], "unit": "GB/s", "frac": 0.0, "traffic": None, "kernel": "k_rollout",
                    "ms_per_launch": ro_ms / max(ro_n, 1), "note": "rollouts are integer-issue bound in registers: 0 algorithmic HBM bytes "
                    "(SURVEY §8d); board steps/s = %.3g" % (pdelta["rollout_steps"] / max(ro_ms / 1e3, 1e-9))}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline(cfg["workload_key"], sims, args.cpu_seconds)
            except Exception as ex:   # the oracle/_ref modules are prebuilt; report rather than die
                cpu = {"value": None, "unit": "sims/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
        config = dict(cfg["config"])
        config["path_cache"] = ("on: the children's statistics of every trace level are kept next to the trace, the next walk serves the levels it shares with it "
                                "from there (b200_set_path_cache; results identical, tests/test_gpu_engine.py::test_path_cache_*); %.1f %% of the walked levels"
                                % (100.0 * delta.get("cached_levels", 0) / max(delta["trace_levels"], 1))) if eng_path_cache else "off"
        config.update({"parallelism": "games sharded x%d, no data-path collective in the search; one exchange step per move (replay rows, all-gather)" % world,
                       "l2": "inputs larger than L2: %.1f GB of arenas per GPU; %.2f GB of activations stream through L2 every sim-step"
                             % (G * M * ARENA_BYTES_PER_SLOT / 1e9, G * 7 * 1792 * 4 / 1e9)})
        out = {"metric": "mcts_sims_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": config, "roofline": roof, "roofline_select_backup": roof_tree, "cpu_baseline": cpu,
               "e2e": {"value": e2e_sims / e2e_s, "unit": "sims/s", "h2d_bytes_per_step": G * 80 * world, "d2h_bytes_per_step": G * (4 + 84 + 80) * world,
                       "ms_per_step": 1e3 * e2e_s / steps, "includes": "set_games (H2D) + play_move (D2H actions, stats, status) + get_games (D2H) + replay drain + all-gather"},
               "same_workload": {"value_pass_vs_instrumented_vs_e2e": bool(same), "keys": list(WORK_KEYS),
                                 "differing": {k: [delta[k], pdelta[k], edelta[k]] for k in WORK_KEYS if not (delta[k] == pdelta[k] == edelta[k])},
                                 "how": "three identical engines built from the same seeds, W warm-up moves, then the same K moves (deterministic search)"},
               "gpu_launches": int(launches), "clocks": clk.summary(), "trajectory_allgather": traj,
               "phases_ms_per_step": {k: v[0] / steps for k, v in phases.items()}, "instrumented_ms_per_step": ms_instr / steps,
               "phases_note": "value / ms_per_step: K steps on the production path (each simulation step replayed as one CUDA graph).  phases_ms_per_step, "
                              "roofline.*: the same K steps on a second identical engine with an event pair around every kernel (direct launches), "
                              "instrumented_ms_per_step long",
               "counters_per_step": {k: v / steps for k, v in delta.items()}, "longest_trace_last_step": longest_trace}
    # ---- BASELINE configs[1] alongside (Vanilla MCTS, random rollouts, no value net): short, so it rides in the same line.  A Vanilla
    # episode on this environment is short and front-loaded: the CLT policy commits to ONE line of play within ~4 moves, from then on
    # nearly every simulation walks the kept tree to a terminal node and rolls nothing out (the CPU oracle shows the same: 40 / 28 / 13 / 2 /
    # <0.1 playout steps per simulation on moves 0 / 1 / 2 / 3 / 4+, game over after ~37 moves).  Timing moves W.. of a running game (round 1)
    # therefore measured almost no k_rollout work.  The line now times WHOLE EPISODES from fresh games (every phase in its natural share)
    # and reports the rollout-heavy opening (moves 0-2, where k_rollout's integer-issue-bound playouts dominate) separately.
    if cfg["mode"] == "lp" and not args.no_secondary:
        G2, sims2, ep_moves, open_moves = 4096, 300, 40, 3

        def vanilla_engine():
            e = BatchedEngine(G2, max_nodes=8192, mode="vanilla", eval_kind="synthetic", env_args=ENV_ARGS, seed=BASE_SEED + 7919 * rank,
                              device=local_rank, rollout_variance=1e3, overflow_reset=True)
            e.set_games(PT.new_games(G2, ENV_ARGS, D.shard_seeds(BASE_SEED, G2 * world, rank, world)))
            e.set_gc_headroom(8192 * 5 // 32)
            return e
        e2 = vanilla_engine()                      # warm-up on a throwaway engine (kernels loaded, clocks up), then fresh games
        for _ in range(max(args.warmup, 3)):
            e2.play_move(sims2, auto_reset=True, want_stats=False)
        e2.close()
        e2 = vanilla_engine()
        k0 = e2.counters()
        D.barrier()
        torch.cuda.synchronize()
        e2.timer_start()
        for _ in range(open_moves):
            e2.play_move(sims2, auto_reset=True, want_stats=False)
        ms_open = D.max_over_ranks(e2.timer_stop(), dev)
        ko = e2.counters()
        e2.timer_start()
        for _ in range(ep_moves - open_moves):
            e2.play_move(sims2, auto_reset=True, want_stats=False)
        ms2 = ms_open + D.max_over_ranks(e2.timer_stop(), dev)
        k1 = e2.counters()
        d2 = D.sum_over_ranks({k: k1[k] - k0[k] for k in k1 if k != "max_trace_len"}, dev)
        do = D.sum_over_ranks({k: ko[k] - k0[k] for k in ko if k != "max_trace_len"}, dev)
        e2.close()
        if out is not None:
            out["also_configs1_vanilla"] = {"workload": "BASELINE configs[1]: Vanilla MCTS, %d games/GPU, %d sims/move, whole episodes from fresh games (%d moves)"
                                                        % (G2, sims2, ep_moves),
                                            "value": d2["sims"] / (ms2 / 1e3), "unit": "sims/s", "ms_per_step": ms2 / ep_moves, "moves_timed": ep_moves,
                                            "rollout_steps_per_sim": d2["rollout_steps"] / max(d2["sims"], 1),
                                            "mean_trace_len": d2["trace_levels"] / max(d2["sims"], 1), "games_finished": d2["games_finished"],
                                            "opening_moves_0_2": {"value": do["sims"] / (ms_open / 1e3), "unit": "sims/s", "ms_per_step": ms_open / open_moves,
                                                                  "rollout_steps_per_sim": do["rollout_steps"] / max(do["sims"], 1),
                                                                  "board_steps_per_sec": (do["rollout_steps"] + 7 * do["expansions"]) / (ms_open / 1e3),
                                                                  "mean_trace_len": do["trace_levels"] / max(do["sims"], 1),
                                                                  "bound": "k_rollout: integer issue (in-register playouts, 0 HBM bytes), SURVEY 8d"}}
    # ---- BASELINE configs[3] proper (65536 games over 8 GPUs = 8192 per GPU) and configs[4] (distributional head, 16384 games over 8 GPUs =
    # 2048 per GPU, 1500 sims/move): the per-GPU shares, a few moves each, so that the default line carries every BASELINE configuration
    if cfg["mode"] == "lp" and not args.no_secondary and cfg["games_per_gpu"] == 16384:
        def short_run(tag, label, n_games, n_sims, max_nodes, mode, eval_kind, w=None, dw=None, moves=3, warm=3):
            e3 = BatchedEngine(n_games, max_nodes=max_nodes, mode=mode, eval_kind=eval_kind, weights=w, dist_weights=dw, env_args=ENV_ARGS,
                               seed=BASE_SEED + 7919 * rank, device=local_rank, overflow_reset=True)
            e3.set_games(PT.new_games(n_games, ENV_ARGS, D.shard_seeds(BASE_SEED, n_games * world, rank, world)))
            e3.set_gc_headroom(max_nodes * 5 // 32)
            for _ in range(warm):
                e3.play_move(n_sims, auto_reset=True, want_stats=False)
            q0 = e3.counters()
            D.barrier()
            torch.cuda.synchronize()
            e3.timer_start()
            for _ in range(moves):
                e3.play_move(n_sims, auto_reset=True, want_stats=False)
            ms3 = D.max_over_ranks(e3.timer_stop(), dev)
            q1 = e3.counters()
            d3 = D.sum_over_ranks({k: q1[k] - q0[k] for k in q1 if k != "max_trace_len"}, dev)
            e3.close()
            if out is not None:
                out[tag] = {"workload": label, "value": d3["sims"] / (ms3 / 1e3), "unit": "sims/s", "ms_per_step": ms3 / moves, "moves_timed": moves,
                            "warmup_moves": warm, "mean_trace_len": d3["trace_levels"] / max(d3["sims"], 1), "tree_resets_per_step": d3["tree_resets"] / moves}
        short_run("also_configs3_8192_games_per_gpu", "BASELINE configs[3] per-GPU share: ValueSimLP + value net (net_tc), 8192 games/GPU (65536 over 8 GPUs), 500 sims/move",
                  8192, 500, 16384, "lp", cfg["eval"], w=weights)
        from tetris_mcts_b200.agents.DistValueSimOnline import init_dist_weights
        short_run("also_configs4_distributional", "BASELINE configs[4] per-GPU share: distributional head (agents/core_distributional.py; network on tcgen05: "
                  "k_tdc_conv / k_tdc_fc), 2048 games/GPU (16384 over 8 GPUs), 1500 sims/move", 2048, 1500, 32768, "dist", cfg["eval"],
                  dw=init_dist_weights(0, 50), moves=2, warm=2)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="valuesimlp", choices=["valuesimlp", "vanilla", "dist"])
    ap.add_argument("--games-per-gpu", type=int, default=None)
    ap.add_argument("--sims", type=int, default=None)
    ap.add_argument("--max-nodes", type=int, default=None)
    ap.add_argument("--gc-headroom", type=int, default=None, help="collect between moves every game with fewer free slots (default 5/32 of max_nodes; 0 = lazy collection only)")
    ap.add_argument("--eval", default=os.environ.get("B200_EVAL", "net_tc"), choices=["net", "net_tc", "synthetic"])
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--path-cache", default="auto", choices=["auto", "on", "off"],
                    help="b200_set_path_cache (memory traffic only, results identical): auto = the engine's default where it applies (LP mode, max_nodes <= 65536)")
    ap.add_argument("--ref-moves-per-step", type=int, default=2)
    ap.add_argument("--exchange-rows", type=int, default=131072, help="rows (212 B) of the fixed-size replay block each rank contributes to the per-move all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's actions and the games it left (get_games) as float64 DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200 and --steps >= 1")
    if args.workload == "vanilla":
        G, sims, M, mode = args.games_per_gpu or 4096, args.sims or 300, args.max_nodes or 8192, "vanilla"
        name = "BASELINE configs[1]: Vanilla MCTS (random rollouts, no value net), %d games/GPU, %d sims/move" % (G, sims)
    elif args.workload == "dist":
        G, sims, M, mode = args.games_per_gpu or 2048, args.sims or 1500, args.max_nodes or 32768, "dist"
        name = "BASELINE configs[4]: distributional head (agents/core_distributional.py), %d games/GPU (16384 over 8 GPUs), %d sims/move" % (G, sims)
    else:
        G, sims, M, mode = args.games_per_gpu or 16384, args.sims or 500, args.max_nodes or 16384, "lp"
        name = "BASELINE configs[2]: ValueSimLP + value net, %d games/GPU, %d sims/move" % (G, sims)
    headroom = args.gc_headroom if args.gc_headroom is not None else M * 5 // 32
    cfg = dict(games_per_gpu=G, sims=sims, max_nodes=M, mode=mode, eval=args.eval, workload_key=args.workload, gc_headroom=headroom,
               config={"workload": name, "games_per_gpu": G, "sims_per_move": sims, "max_nodes": M, "evaluator": args.eval if mode != "vanilla" else "rollout",
                       "env_args": "((20,10),1,0,0)", "weights": "default-init distribution, numpy PCG64 seed 0",
                       "garbage_collection": "TreeAgent.remove_nodes() between moves for every game with fewer than %d free slots, batched over the games "
                                             "(b200_set_gc_headroom; reference equivalent: the driver calling agent.remove_nodes(), agents/agent.py:246-257), "
                                             "plus the reference's own call inside new_node when a free list runs dry in the middle of a move" % headroom,
                       "arena_overflow": "reference semantics up to max_nodes per game; a game whose reachable set fills its arena (a collection recovers fewer "
                                         "than max_nodes/8 slots; the reference then collects at nearly every expansion and dies with IndexError) drops its tree "
                                         "and re-roots (counters_per_step.tree_resets)"})
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_b200(args, cfg)


if __name__ == "__main__":
    main()
