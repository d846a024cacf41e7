"""The device board-step header (tetris_mcts_b200/csrc/tetris_dev.cuh) compiled for the HOST with g++ (tests/host_env_shim.cpp)
and run against the oracle (oracle/tetris_oracle.c, SPEC_PYTETRIS.md) on random action sequences: the same source the kernels
compile, checked bit for bit without a GPU (records, scores, line statistics, bag/RNG state, observation keys).  The GPU suite
repeats the comparison through the C-ABI (tests/test_gpu_env.py)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


@pytest.fixture(scope="module", params=[()], ids=["default"])
def host_env(request, tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostenv") / "host_env.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", *request.param, "-I", os.path.join(ROOT, "tetris_mcts_b200", "csrc"),
                    os.path.join(HERE, "host_env_shim.cpp"), "-o", so], check=True)
    return C.CDLL(so)


@pytest.mark.parametrize("env_args", [(1, 0, 0), (1, 1, 1), (2, 0, 1), (3, 1, 0), (1, 0, 1), (1, 1, 0), (2, 1, 1), (4, 0, 0)])
def test_device_header_steps_like_the_oracle(host_env, env_args):
    import oracle_py as O
    app, scoring, randomizer = env_args
    rng = np.random.default_rng(11 + app)
    n = 1024
    recs = O.fresh_records(n, 1000, app, scoring, randomizer)
    hard_drops = 0
    for step in range(300):
        p = [0.1, 0.1, 0.1, 0.1, 0.1, 0.35, 0.15] if step % 2 else [1 / 7] * 7   # every other step is rich in hard drops
        a = rng.choice(7, size=n, p=p).astype(np.int32)
        if step % 10 == 3:
            a[::9] = 7                                                              # VanillaC.py:7 draws randint(0, 7): an id outside 0..6 is a no-op
        want = O.play_records(recs, a)
        got = recs.copy()
        host_env.host_play_records(got.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p), n)
        assert np.array_equal(want, got), (env_args, step)
        hard_drops += int((a == 5).sum())
        recs = want
        if step % 25 == 0:                                                          # observation keys, finished games included
            keys = np.zeros((n, 12), np.uint32)
            host_env.host_obskeys(recs.ctypes.data_as(C.c_void_p), keys.ctypes.data_as(C.c_void_p), n)
            for i in range(0, n, 5):
                assert np.array_equal(keys[i], O.Game(record=recs[i]).obskey()), (env_args, step, i)
        ended = ((recs[:, 10] >> 21) & 1).astype(bool)
        if ended.any() and step % 50 == 49:                                         # keep the population alive
            recs[ended] = O.fresh_records(int(ended.sum()), 5000 + step, app, scoring, randomizer)
    assert hard_drops > 10000
    keys = np.zeros((n, 12), np.uint32)
    host_env.host_obskeys(recs.ctypes.data_as(C.c_void_p), keys.ctypes.data_as(C.c_void_p), n)
    for i in range(0, n, 37):
        assert np.array_equal(keys[i], O.Game(record=recs[i]).obskey())
