"""Arena growth + first timings (development aid)."""
import os, sys, time
import numpy as np
sys.path.insert(0, '.')
from tetris_mcts_b200 import pyTetris as PT
from tetris_mcts_b200.engine import BatchedEngine
from tetris_mcts_b200.model.model_vv import init_weights
G, M, sims = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
moves = int(sys.argv[4]); ev = sys.argv[5] if len(sys.argv) > 5 else 'net'
eng = BatchedEngine(G, max_nodes=M, mode='lp', eval_kind=ev, weights=init_weights(0), overflow_reset=True)
eng.set_games(PT.new_games(G, (1, 0, 0), np.arange(123, 123 + G, dtype=np.uint32)))
eng.set_gc_headroom(int(os.environ.get('GC_HEADROOM', '0')))
TIMING = os.environ.get('NO_TIMING') != '1'
eng.set_timing(TIMING)
prev = eng.counters()
pprev = {k: v[0] for k, v in eng.phase_ms().items()} if TIMING else None
for mv in range(moves):
    t = time.time()
    try:
        eng.play_move(sims, True, False)
    except Exception as e:
        print('move', mv, 'ERR', e); break
    dt = time.time() - t
    c = eng.counters()
    d = {k: c[k] - prev[k] for k in c}; prev = c
    ph = ''
    if TIMING:
        pm = {k: v[0] for k, v in eng.phase_ms().items()}
        ph = ' | ms: ' + ' '.join('%s %.1f' % (k[:6], pm[k] - pprev[k]) for k in ('select_expand', 'conv', 'fc', 'backup', 'gc'))
        pprev = pm
    print('move %2d %.3fs sims/s %.3g new_nodes/game %.0f evals/sim %.2f D %.2f Dmax %d gcs %d resets %d finished %d%s' % (
        mv, dt, G * sims / dt, d['new_nodes'] / G, d['eval_requests'] / max(d['sims'], 1), d['trace_levels'] / max(d['sims'], 1), c['max_trace_len'],
        d['gcs'], d['tree_resets'], c['games_finished'], ph), flush=True)
print({k: (round(v[0], 2), v[1]) for k, v in eng.phase_ms().items()})
try:
    from tetris_mcts_b200 import _lib as _L
    tl = np.zeros(G, np.int32)
    _L.lib().b200_debug_trace_lens.argtypes = [_L.P, _L.P]
    _L.check(_L.lib().b200_debug_trace_lens(eng.h, _L.ptr(tl)))
    print('trace length of the last simulation over the games: mean %.1f  percentiles 50/75/90/95/98/99/99.9/100 = %s' % (
        tl.mean(), [int(x) for x in np.percentile(tl, [50, 75, 90, 95, 98, 99, 99.9, 100])]))
except Exception as ex:
    print('trace lens unavailable', ex)

import ctypes
from tetris_mcts_b200 import _lib as L
pr = np.zeros(16, np.uint64)
L.lib().b200_debug_prof.argtypes = [L.P, L.P]
L.check(L.lib().b200_debug_prof(eng.h, L.ptr(pr)))
names = ['S0_arrive', 'wait_c1', 'E1', 'wait_c2', 'E2', 'wait_c3', 'E3', 'S0_wait_key', 'iss_wait_a0', 'iss_conv1', 'iss_wait_a1', 'iss_conv2', 'iss_wait_a2', 'iss_conv3', 'S0_compute', 'S0_fence']
tot = pr[:8].sum() + pr[14:16].sum()
print({n: round(float(pr[i]) / max(float(tot), 1), 3) for i, n in enumerate(names)}, 'worker cycles total', int(tot), 'boards', c['eval_requests'] // 148)

pt = np.zeros(16, np.uint64)
L.lib().b200_debug_prof_tree.argtypes = [L.P, L.P]
L.check(L.lib().b200_debug_prof_tree(eng.h, L.ptr(pt)))
tt = float(pt[:4].sum())
print('k_select_expand sampled groups', int(pt[4]), {n: round(float(pt[i]) / max(tt, 1), 3) for i, n in enumerate(['select', 'leaf_load', 'expand', 'finish+evalreq'])}, 'mean clk/group', int(tt / max(float(pt[4]), 1)))
