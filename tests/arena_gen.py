"""Seeded synthetic search arenas in the reference's array layout (agents/agent.py:58-88), per SURVEY §8(d):
7-ary, depth 4-12, visit in [1,1000], value ~ U(0,50), variance ~ U(1,100), score non-decreasing along edges,
10-30 % duplicated observations among siblings."""
import zlib

import numpy as np


def make_arena(seed, M=4096, max_depth=8, p_expand=0.6, p_dup=0.2, p_zero_child=0.1, unvisited=0.0, single_low=False):
    rng = np.random.default_rng(seed)
    child = np.zeros((M, 7), np.int32)
    score = np.zeros(M, np.float32)
    n2o = np.zeros(M, np.int32)
    depth = np.zeros(M, np.int32)
    nxt, nobs = 2, 2
    n2o[1] = 1
    score[1] = float(rng.integers(0, 500))
    frontier = [1]
    while frontier:
        n = frontier.pop(0)
        if depth[n] >= max_depth or nxt + 7 >= M:
            continue
        if n != 1 and rng.random() > p_expand:
            continue
        sib_obs = []
        for a in range(7):
            if rng.random() < p_zero_child:
                continue
            c = nxt
            nxt += 1
            child[n, a] = c
            depth[c] = depth[n] + 1
            score[c] = score[n] + float(rng.choice([0, 0, 0, 1, 2, 34, 100, 300]))
            if sib_obs and rng.random() < p_dup:
                n2o[c] = sib_obs[rng.integers(0, len(sib_obs))]
            else:
                n2o[c] = nobs
                nobs += 1
            sib_obs.append(n2o[c])
            frontier.append(c)
        if child[n].any() and rng.random() < 0.15:   # the same child in two slots
            nz = np.nonzero(child[n])[0]
            z = np.nonzero(child[n] == 0)[0]
            if len(z):
                child[n, z[0]] = child[n, nz[0]]
    visit = np.zeros(M, np.int32)
    value = np.zeros(M, np.float32)
    variance = np.zeros(M, np.float32)
    visit[1:nobs] = rng.integers(1, 1001, nobs - 1)
    value[1:nobs] = rng.uniform(0, 50, nobs - 1).astype(np.float32)
    variance[1:nobs] = rng.uniform(1, 100, nobs - 1).astype(np.float32)
    if unvisited > 0:
        mask = rng.random(nobs) < unvisited
        mask[:2] = False
        if single_low:   # at most one low observation per sibling set, so rand() % 1 == 0 whatever rand() returns
            for n in range(1, nxt):
                obs = sorted(set(int(n2o[c]) for c in child[n] if c))
                low = [o for o in obs if mask[o]]
                for o in low[1:]:
                    mask[o] = False
        idx = np.nonzero(mask)[0]
        visit[idx] = 0
        value[idx] = 0
        variance[idx] = 0
    return dict(child=child, visit=visit, value=value, variance=variance, score=score, n2o=n2o, n_nodes=nxt, n_obs=nobs)


def near_tie_arena(seed, M=64):
    """Root with seven children whose CLT scores differ in the last float bits: exercises core.h:94-101 rounding."""
    rng = np.random.default_rng(seed)
    a = dict(child=np.zeros((M, 7), np.int32), visit=np.zeros(M, np.int32), value=np.zeros(M, np.float32),
             variance=np.zeros(M, np.float32), score=np.zeros(M, np.float32), n2o=np.zeros(M, np.int32))
    a["n2o"][1] = 1
    a["score"][1] = 17.0
    base_v = np.float32(rng.uniform(10, 40))
    for i in range(7):
        c = 2 + i
        a["child"][1, i] = c
        a["n2o"][c] = 2 + i
        a["score"][c] = 17.0 + float(rng.integers(0, 3))
        a["visit"][2 + i] = int(rng.integers(5, 9))
        a["value"][2 + i] = np.nextafter(base_v, np.float32(100), dtype=np.float32) if rng.random() < 0.5 else base_v
        a["variance"][2 + i] = np.float32(rng.choice([4.0, 4.0000005, 3.9999998]))
    a["visit"][1] = 50
    a["n_nodes"], a["n_obs"] = 9, 9
    return a


def arena_crc(a):
    """CRC-32 of an arena's arrays: ties a golden that stores only a seed to the exact arena the seed regenerates."""
    return zlib.crc32(b"".join(np.ascontiguousarray(a[k]).tobytes() for k in ("child", "visit", "value", "variance", "score", "n2o")))


def boards(n, seed):
    """tools/test.py:23-28 style inputs for the value network: random {0,1} cells, top rows cleared, four -1 cells."""
    rng = np.random.default_rng(seed)
    b = (rng.random((n, 20, 10)) < 0.45).astype(np.int8)
    for i in range(n):
        b[i, :rng.integers(2, 12)] = 0
        r, c = rng.integers(0, 3), rng.integers(0, 8)
        b[i, r:r + 2, c:c + 2] = -1
    return b


def state_to_obskey(s):
    """int8[20,10] observation -> SPEC §6 observation key (test helper for the synthetic evaluator)."""
    key = np.zeros(12, np.uint32)
    cells = []
    for r in range(20):
        row = 0
        for c in range(10):
            if s[r, c] == 1:
                row |= 1 << c
            elif s[r, c] == -1:
                cells.append(r * 10 + c)
        key[r >> 1] |= np.uint32(row << ((r & 1) * 16))
    cells.sort()
    key[10] = np.uint32(sum(v << (8 * i) for i, v in enumerate(cells[:4])))
    return key


def golden_bk_dist(z, p):
    """node_dist after the backup of tests/golden/dist_golden.npz case prefix p: stored whole (bk_dist), or as the rows the backup
    changed (bk_rows, bk_dist_rows) on top of the stored input node_dist."""
    if p + "bk_dist" in z:
        return z[p + "bk_dist"]
    bk = z[p + "node_dist"].copy()
    bk[z[p + "bk_rows"]] = z[p + "bk_dist_rows"]
    return bk


def make_dist_arena(seed, M=512, bins=50, max_depth=6, unvisited=0.0):
    """Seeded node-indexed arena for the distributional cores: node_stats f32[M,5] = {visit, mean, reward, variance, M2},
    node_dist f32[M,bins] (rows sum to 1), child int32[M,7] (agents/core_distributional.py)."""
    a = make_arena(seed, M=M, max_depth=max_depth, p_dup=0.0)
    rng = np.random.default_rng(seed + 7)
    n = a["n_nodes"]
    ns = np.zeros((M, 5), np.float32)
    ns[1:n, 0] = rng.integers(1, 400, n - 1)
    ns[1:n, 1] = rng.uniform(0, 800, n - 1)
    ns[:, 2] = a["score"]
    ns[1:n, 3] = rng.uniform(1, 5000, n - 1)
    ns[1:n, 4] = ns[1:n, 3] * np.maximum(ns[1:n, 0] - 1, 1)
    if unvisited > 0:
        m = rng.random(M) < unvisited
        m[:2] = False
        ns[m, 0] = 0
    nd = rng.random((M, bins)).astype(np.float32) ** 4
    nd /= nd.sum(axis=1, keepdims=True)
    return dict(child=a["child"], node_stats=ns, node_dist=nd.astype(np.float32), n_nodes=n)
