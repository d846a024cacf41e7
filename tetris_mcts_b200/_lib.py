"""ctypes binding of libb200_tetris_mcts.so (include/b200_tetris_mcts.h).  There is no fallback: if the library is
missing or no CUDA device is present, the calls raise."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200_TETRIS_LIB") or os.path.join(HERE, "libb200_tetris_mcts.so")   # the variable is a development aid (A/B builds)

REC_WORDS = 20
KEY_WORDS = 12
N_ACTIONS = 7
N_WEIGHTS = 478342

MODE_LP, MODE_SINGLE, MODE_VANILLA, MODE_DIST = 0, 1, 2, 3
EVAL_SYNTHETIC, EVAL_NET, EVAL_NET_TC = 0, 1, 2
ERR_NAMES = {1: "BAD_ARG", 2: "CUDA", 3: "ARENA_FULL", 4: "TRACE_FULL", 5: "NO_WEIGHTS"}


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("b200 error %d (%s): %s" % (code, ERR_NAMES.get(code, "?"), msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("n_games", C.c_int32), ("max_nodes", C.c_int32), ("mode", C.c_int32), ("low", C.c_int32),
                ("lp_end_from_obs", C.c_int32), ("lp_var_gamma2", C.c_int32), ("stale_pop", C.c_int32), ("overflow_reset", C.c_int32),
                ("eval_kind", C.c_int32), ("trace_max", C.c_int32), ("actions_per_drop", C.c_int32),
                ("scoring", C.c_int32), ("randomizer", C.c_int32), ("device", C.c_int32), ("seed", C.c_uint32),
                ("gamma", C.c_double), ("rollout_variance", C.c_double), ("dist_bins", C.c_int32), ("dist_vmin", C.c_double), ("dist_vmax", C.c_double)]


_lib = None
P = C.c_void_p


def lib():
    """Load the CUDA library; raise (loudly) if it has not been built — the product has no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python -m tetris_mcts_b200.build` (nvcc, sm_100a). "
                              "tetris_mcts_b200 has no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.b200_last_error.restype = C.c_char_p
        L.b200_engine_create.argtypes = [C.POINTER(Config), C.POINTER(P)]
        L.b200_engine_destroy.argtypes = [P]
        L.b200_engine_set_stream.argtypes = [P, P]
        L.b200_engine_get_stream.argtypes = [P, C.POINTER(P)]
        L.b200_load_weights.argtypes = [P, P]
        L.b200_set_games.argtypes = [P, P]
        L.b200_get_games.argtypes = [P, P]
        L.b200_update_root.argtypes = [P, C.c_int]
        L.b200_run_sims.argtypes = [P, C.c_int]
        L.b200_get_stats.argtypes = [P, P, P]
        L.b200_env_step.argtypes = [P, P]
        L.b200_play_move.argtypes = [P, C.c_int, C.c_int, P, P]
        L.b200_status.argtypes = [P, P]
        L.b200_finished_games.argtypes = [P, P, C.c_int, P]
        L.b200_remove_nodes.argtypes = [P, C.c_int]
        L.b200_set_gc_headroom.argtypes = [P, C.c_int]
        L.b200_set_path_cache.argtypes = [P, C.c_int]
        L.b200_counters.argtypes = [P, P]
        L.b200_sync.argtypes = [P]
        L.b200_set_timing.argtypes = [P, C.c_int]
        L.b200_timer_start.argtypes = [P]
        L.b200_timer_stop.argtypes = [P, P]
        L.b200_phase_ms.argtypes = [P, P, P]
        L.b200_export_game.argtypes = [P, C.c_int] + [P] * 13
        L.b200_valuenet_forward.argtypes = [P, P, C.c_int, P, P]
        L.b200_debug_act3.argtypes = [P, P, C.c_int, P]
        L.b200_tetris_step.argtypes = [P, P, C.c_int]
        L.b200_tetris_new.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int]
        L.b200_tetris_state.argtypes = [P, P, C.c_int]
        L.b200_select_trace_obs.argtypes = [C.c_int] + [P] * 6 + [C.c_int, C.c_int, P, P, C.c_int, P]
        L.b200_backup_trace_obs.argtypes = [P, C.c_int] + [P] * 5 + [C.c_int, C.c_double, C.c_double, C.c_double]
        L.b200_backup_trace_obs_LP.argtypes = ([P, C.c_int] + [P] * 6 + [C.c_int, P, P, C.c_int, P, P, C.c_double,
                                               C.c_int, C.c_int])
        L.b200_get_unique_child_obs.argtypes = [C.c_int, P, P, P, C.c_int, P, P, P]
        L.b200_get_all_childs.argtypes = [C.c_int, P, C.c_int, P]
        L.b200_collect_samples_dev.argtypes = [P, C.c_int, P, C.c_int, P]
        L.b200_replay_enable.argtypes = [P, C.c_int, C.c_int]
        L.b200_replay_drain_dev.argtypes = [P, P, C.c_int, P]
        L.b200_replay_policy.argtypes = [P, C.c_int, C.c_int, C.c_int]
        L.b200_replay_policy_step.argtypes = [P, C.c_int64, P, P]
        L.b200_replay_policy_trained.argtypes = [P, C.c_int64]
        L.b200_replay_peek_dev.argtypes = [P, P, C.c_int]
        L.b200_replay_append.argtypes = [P, P, C.c_int]
        L.b200_load_dist_weights.argtypes = [P, P, C.c_int]
        L.b200_distnet_forward.argtypes = [P, P, C.c_int, C.c_int, P]
        L.b200_export_dist.argtypes = [P, C.c_int, P, P]
        L.b200_dist_shift_distribution.argtypes = [P, C.c_int, C.c_double, C.c_double, C.c_double, P]
        L.b200_dist_mean_variance.argtypes = [P, C.c_int, C.c_double, C.c_double, P, P]
        L.b200_dist_select_trace.argtypes = [C.c_int, P, P, C.c_int, C.c_int, P, P, C.c_int, P]
        L.b200_dist_backup_trace.argtypes = [P, C.c_int, P, P, C.c_int, C.c_int, C.c_double, P, C.c_double, C.c_double]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise B200Error(rc, lib().b200_last_error().decode())


def ptr(a):
    return None if a is None else a.ctypes.data_as(P)


def exported_symbols():
    """Names declared in include/b200_tetris_mcts.h (used by the CPU-side ABI test)."""
    import re
    hdr = os.path.join(HERE, "..", "include", "b200_tetris_mcts.h")
    txt = open(hdr).read()
    return sorted(set(re.findall(r"\b(b200_[a-z_A-Z0-9]+)\s*\(", txt)))
