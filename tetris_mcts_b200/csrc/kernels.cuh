// kernels.cuh — the __global__ entry points of the engine (sm_100a).  Launch geometry: one 8-lane group per game,
// 128-thread blocks (16 games per block), so G games = G/16 blocks; at G >= 16384 that is >= 1024 blocks = ~7 CTAs
// per SM on 148 SMs.  The tree walk is pointer chasing (latency bound); occupancy, not ILP, hides HBM latency here.
#pragma once
#include "search_dev.cuh"

namespace b200 {

constexpr int GROUPS_PER_BLOCK = 16;
constexpr int TPB = GROUPS_PER_BLOCK * 8;
constexpr int SE_GAMES_PER_BLOCK = GROUPS_PER_BLOCK;   // k_select_expand: four games per warp

__device__ __forceinline__ void load_rec(const uint32_t *src, uint32_t (&w)[REC_WORDS]) {
#pragma unroll
    for (int q = 0; q < REC_WORDS / 4; ++q) {
        uint4 v = reinterpret_cast<const uint4 *>(src)[q];
        w[q * 4] = v.x; w[q * 4 + 1] = v.y; w[q * 4 + 2] = v.z; w[q * 4 + 3] = v.w;
    }
}
__device__ __forceinline__ void store_rec(uint32_t *dst, const uint32_t (&w)[REC_WORDS]) {
#pragma unroll
    for (int q = 0; q < REC_WORDS / 4; ++q)
        reinterpret_cast<uint4 *>(dst)[q] = make_uint4(w[q * 4], w[q * 4 + 1], w[q * 4 + 2], w[q * 4 + 3]);
}

// ---------------------------------------------------------------- arena initialisation (agent.py:58-88)
__global__ void k_init_arena(Arena A, const uint32_t *default_rec, uint32_t seed) {
    size_t n = (size_t)A.G * A.M;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        int g = (int)(i / A.M), idx = (int)(i % A.M);
        uint32_t w[REC_WORDS];
#pragma unroll
        for (int q = 0; q < REC_WORDS; ++q) w[q] = default_rec[q];      // agent.py:70 every slot starts as env(*env_args)
        store_rec(A.rec + i * REC_WORDS, w);
        if (idx < A.M - 1) { A.nfree[i] = idx + 1; A.ofree[i] = idx + 1; }   // agent.py:72 deque(range(1, M))
        if (idx == 0) {
            A.n_nfree[g] = A.M - 1; A.n_ofree[g] = A.M - 1;
            A.root[g] = 0; A.episode[g] = 0; A.status[g] = ST_OK;
            uint32_t s = seed + 0x9E3779B9u * (uint32_t)(g + 1);
            A.srng[g] = s ? s : 0x2545F491u;
        }
    }
}

// ---------------------------------------------------------------- batched board step (SPEC §3, play.py:150)
__global__ void k_env_step(uint32_t *recs, const int32_t *actions, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[REC_WORDS];
    load_rec(recs + (size_t)i * REC_WORDS, w);
    Game g;
    unpack(g, w);
    play(g, actions[i]);
    pack(g, w);
    store_rec(recs + (size_t)i * REC_WORDS, w);
}

// observation int8[20,10] of packed games (SPEC §1; agent.py:116 getState())
__global__ void k_env_state(const uint32_t *recs, int8_t *out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[REC_WORDS];
    load_rec(recs + (size_t)i * REC_WORDS, w);
    Game g;
    unpack(g, w);
    uint32_t k[KEY_WORDS];
    obskey(g, k);
    int8_t *o = out + (size_t)i * 200;
    for (int r = 0; r < 20; ++r) {
        uint32_t row = (k[r >> 1] >> ((r & 1) * 16)) & 0x3ffu;
        for (int c = 0; c < 10; ++c) o[r * 10 + c] = (int8_t)((row >> c) & 1u);
    }
    for (int j = 0; j < 4; ++j) o[(k[10] >> (8 * j)) & 0xffu] = -1;
}

__device__ __forceinline__ void reset_game(Game &g) {   // SPEC §4 reset(): keeps the RNG stream
#pragma unroll
    for (int i = 0; i < 10; ++i) g.w[i] = 0;
    g.bag = 0x7fu; g.dropcnt = 0; g.end = 0; g.combo = 0; g.score = 0; g.lines = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) g.ls[i] = 0;
    spawn(g);
}

// ---------------------------------------------------------------- suspension for garbage collection
// A group that finds its free list empty queues its game for k_gc and records what to redo afterwards.
__device__ __forceinline__ void suspend_for_gc(const Arena &A, const Grp &gp, int g, int what, int a) {
    if (gp.lane == 0) {
        A.pending[g] = what; A.resume_a[g] = a;
        A.gc_list[atomicAdd(A.n_req + 1, 1)] = g;
    }
}

// queue the evaluation requests of one group: lanes whose bit is set in `need` ask for observation my_o, slot = lane
__device__ __forceinline__ void emit_requests(const Arena &A, const Grp &gp, int g, unsigned need, int my_o) {
    if (need == 0) return;
    int base = 0;
    if (gp.lane == 0) { base = atomicAdd(A.n_req, __popc(need)); atomicAdd(&A.counters[2], (unsigned long long)__popc(need)); }
    base = gp.bcast(base, 0);
    if ((need >> gp.lane) & 1u)
        A.req[base + __popc(need & ((1u << gp.lane) - 1u))] = make_uint2((uint32_t)g, (uint32_t)my_o | ((uint32_t)gp.lane << 28));
}

// ---------------------------------------------------------------- update_root (agent.py:296-301)
// auto_reset reproduces play.py:161-177: a finished game is counted, reset and re-rooted.  only_pending: second pass
// after k_gc for the games that had to suspend (the pass is idempotent: see the comments at the two new_node calls).
__global__ void __launch_bounds__(TPB) k_update_root(Arena A, int auto_reset, unsigned long long *game_stats, int only_pending) {
    Grp gp;
    int g = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 3);
    if (g >= A.G) return;
    if (A.pc && gp.lane == 0) A.pc_len[g] = 0;     // path cache: the path starts at another node now
    int status = A.status[g];
    if (only_pending) {
        if (A.pending[g] != PEND_ROOT) return;
        gp.sync();
        if (gp.lane == 0) A.pending[g] = PEND_NONE;
    }
    // overflow_reset: a tree dropped by k_gc (in the last simulation step, or by the collection this very update_root asked for
    // in its first pass) is re-rooted at the live game, then the update proceeds as usual (episode count, auto reset)
    if ((status == ST_ARENA_FULL || status == ST_RESET_DONE) && A.overflow_reset) reset_tree(A, gp, g, status);
    if (status != ST_OK) return;
    const bool may_suspend = !only_pending;
    uint32_t w[REC_WORDS];
    load_rec(A.cur + (size_t)g * REC_WORDS, w);
    int o; float s;
    int idx = new_node(A, gp, g, w, o, s, status, may_suspend);
    if (status == ST_NEED_GC) { suspend_for_gc(A, gp, g, PEND_ROOT, 0); return; }   // nothing was changed yet: redo all
    bool ended = (w[10] >> 21) & 1u;
    if (gp.lane == 0 && status == ST_OK) { A.root[g] = idx; if (ended) A.episode[g] += 1; }
    gp.sync();
    if (ended && auto_reset && status == ST_OK) {
        Game gm;
        unpack(gm, w);
        if (gp.lane == 0 && game_stats) {
            atomicAdd(&game_stats[0], 1ull);
            atomicAdd(&game_stats[1], (unsigned long long)gm.score);
            atomicAdd(&game_stats[2], (unsigned long long)gm.lines);
        }
        if (gp.lane == 0 && A.fin_log) {                       // play.py:164: the line is printed from these numbers before game.reset()
            const int slot = atomicAdd(A.fin_count, 1);
            if (slot < A.fin_cap) reinterpret_cast<int4 *>(A.fin_log)[slot] = make_int4(g, (int)gm.score, (int)gm.lines, A.episode[g]);
        }
        reset_game(gm);
        pack(gm, w);
        if (gp.lane == 0) store_rec(A.cur + (size_t)g * REC_WORDS, w);
        gp.sync();
        idx = new_node(A, gp, g, w, o, s, status, may_suspend);
        // suspended here: the live game is already the fresh one, so the redo pass only re-roots (no second episode++)
        if (status == ST_NEED_GC) { suspend_for_gc(A, gp, g, PEND_ROOT, 0); return; }
        if (gp.lane == 0 && status == ST_OK) A.root[g] = idx;
    }
    if (gp.lane == 0 && status != ST_OK) A.status[g] = status;
}

// After an expansion is complete: which unique children need the network (ValueSimLP.py:55-60 evaluates every unique
// child; core.h:344 only uses results where visit == 0, so only those boards are queued).
__device__ __forceinline__ void request_lp_evals(const Arena &A, const Grp &gp, int g, const Uniq &u, int o) {
    bool ask = u.is_first && A.stat[node_at(A, g, o)].x == 0;
    emit_requests(A, gp, g, gp.ballot(ask), o);
}

// All seven children of `leaf` are linked: de-duplicate the list once (core.h:111-144) and cache it in the row for select.
__device__ __forceinline__ Uniq finish_expansion(const Arena &A, const Grp &gp, int g, int leaf, int c, int o, float s) {
    Uniq u = unique_children(gp, c, o, s);
    A.row[node_at(A, g, leaf) * ROW_WORDS + 24 + gp.lane] = gp.lane < 7 ? (int32_t)link_word(u) : 0;
    return u;
}

// ---------------------------------------------------------------- select + expand (ValueSimLP.py:45-57 etc.)
// What one group hands to the CTA-level epilogue of k_select_expand: its evaluation request (per lane) and its counters.
struct GroupOut { bool ask; int my_o; int sims, D, expanded, new_nodes, cached; };

// The whole warp calls this together (four games per warp): the walk runs in lockstep over the four groups (select_trace, GrpW);
// everything around it is per group.  `g` >= A.G marks a group without a game.
__device__ __forceinline__ void select_expand_group(const Arena &A, const Grp &gp, int g, const float *s_z, uint32_t *stage, GroupOut &out) {
    const bool valid = g < A.G;
    int status = valid ? A.status[g] : ST_ARENA_FULL;
    const bool do_prof = valid && A.prof && (g & 63) == 0 && gp.lane == 0;
    long long ptick = do_prof ? clock64() : 0;
    bool tree_reset = false;
    if (valid && (status == ST_ARENA_FULL || status == ST_RESET_DONE) && A.overflow_reset) { reset_tree(A, gp, g, status); tree_reset = true; }
    const bool active = valid && status == ST_OK;
    ArenaAcc acc(A, valid ? g : 0, s_z);
    if (A.pc && active && !tree_reset && A.mode == MODE_LP) acc.pc_len = A.pc_len[g];   // valid entries of this game's path cache (0 after anything but a backup)
    int D = 0;
#define TREE_PROF(i) do { if (do_prof) { const long long _n = clock64(); atomicAdd(&A.prof[i], (unsigned long long)(_n - ptick)); ptick = _n; } } while (0)
    int leaf = 0;
    if (A.mode == MODE_DIST) {               // grid-uniform branch; the distributional walk keeps its per-group form
        if (active) leaf = dist_select_group(A, gp, g, A.root[g], D, status);
    } else {
        __syncwarp();
        leaf = select_trace(acc, active, active ? A.root[g] : 0, A.low, A.trace_max, D, status, &out.cached);
    }
    if (!active) return;
    if (status != ST_OK) { if (gp.lane == 0) { A.status[g] = status; if (A.pc) A.pc_len[g] = 0; } return; }
    TREE_PROF(0);
    uint32_t w[REC_WORDS];
    load_rec(A.rec + node_at(A, g, leaf) * REC_WORDS, w);
    bool ended = (w[10] >> 21) & 1u;
    int kind = ended ? LEAF_TERMINAL : LEAF_EXPANDED;
    if (do_prof) ptick += (long long)(w[10] & 0u);   // the leaf record has landed
    TREE_PROF(1);
    if (!ended) {
        if (A.mode == MODE_SINGLE || A.mode == MODE_DIST) {   // ValueSim.py:83-88 / DistValueSimOnline.py:66-70: the leaf itself is evaluated
            out.my_o = A.row[node_at(A, g, leaf) * ROW_WORDS + 15];
            out.ask = gp.lane == 7;
        }
        int c, o, a_stop; float s;
        expand_leaf(A, gp, g, leaf, w, c, o, s, status, 0, true, a_stop, stage, &out.new_nodes);
        if (status == ST_NEED_GC) {
            suspend_for_gc(A, gp, g, PEND_EXPAND, a_stop);
            kind = LEAF_SUSPENDED; status = ST_OK;
        } else if (status == ST_OK) {
            TREE_PROF(2);
            out.expanded = 1;
            Uniq u = finish_expansion(A, gp, g, leaf, c, o, s);
            if (A.mode == MODE_LP) {                          // request_lp_evals, queued by the CTA epilogue
                out.ask = u.is_first && A.stat[node_at(A, g, o)].x == 0;
                out.my_o = o;
            }
        }
    }
    if (gp.lane == 0) {
        A.trace_len[g] = D; A.leaf_kind[g] = kind;
        if (status != ST_OK) A.status[g] = status;
        // path cache: entries 0..D-1 describe this trace; the entry of a leaf that was just expanded says "no children" and is dropped;
        // k_backup refreshes the statistics the backup changes and truncates further if a copy went stale (search_dev.cuh "path cache")
        if (A.pc) A.pc_len[g] = (A.mode == MODE_LP && status == ST_OK && kind != LEAF_SUSPENDED) ? (kind == LEAF_EXPANDED ? D - 1 : D) : 0;
    }
    out.sims = 1; out.D = D;
    TREE_PROF(3);
    if (do_prof) atomicAdd(&A.prof[4], 1ull);
#undef TREE_PROF
}

// One launch = one simulation step of every game.  The per-group part is latency bound (pointer chase), so everything that
// would serialise the groups on one address is aggregated per CTA at the end: ONE atomicAdd on the request counter and one per
// statistics counter per CTA (before: ~10 same-address atomics per game per launch, 160 k per launch on two cache lines).
__global__ void __launch_bounds__(TPB, 8) k_select_expand(Arena A) {
    __shared__ __align__(16) float s_z[ZS_N];
    __shared__ __align__(16) uint32_t s_stage[GROUPS_PER_BLOCK * STAGE_GROUP_WORDS];
    __shared__ unsigned s_cnt[6];          // sims, trace levels, expansions, new nodes, longest trace of this CTA, levels served by the path cache
    __shared__ int s_wreq[TPB / 32 + 1];   // requests per warp, then the CTA's base in the request list
    for (int i = threadIdx.x; i < ZS_N / 4; i += TPB) reinterpret_cast<float4 *>(s_z)[i] = reinterpret_cast<const float4 *>(A.ztable)[i];   // (scalar copies were 7 % of the kernel's samples)
    if (threadIdx.x < 6) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    Grp gp;
    const int slot = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 3);
    const int g = slot < A.G ? slot : A.G;                                  // A.G: this group has no game
    GroupOut out{false, 0, 0, 0, 0, 0, 0};
    select_expand_group(A, gp, g, s_z, s_stage + (threadIdx.x >> 3) * STAGE_GROUP_WORDS, out);
    __syncwarp();
    const unsigned askmask = __ballot_sync(0xffffffffu, out.ask);
    if ((threadIdx.x & 31) == 0) s_wreq[threadIdx.x >> 5] = __popc(askmask);
    if (gp.lane == 0 && out.sims) {
        atomicAdd(&s_cnt[0], 1u); atomicAdd(&s_cnt[1], (unsigned)out.D); atomicMax(&s_cnt[4], (unsigned)out.D);
        if (out.expanded) atomicAdd(&s_cnt[2], 1u);
        if (out.new_nodes) atomicAdd(&s_cnt[3], (unsigned)out.new_nodes);
        if (out.cached) atomicAdd(&s_cnt[5], (unsigned)out.cached);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int i = 0; i < TPB / 32; ++i) tot += s_wreq[i];
        s_wreq[TPB / 32] = tot ? atomicAdd(A.n_req, tot) : 0;
        if (tot) atomicAdd(&A.counters[2], (unsigned long long)tot);
        if (s_cnt[0]) { atomicAdd(&A.counters[0], (unsigned long long)s_cnt[0]); atomicAdd(&A.counters[4], (unsigned long long)s_cnt[1]); }
        if (s_cnt[2]) atomicAdd(&A.counters[1], (unsigned long long)s_cnt[2]);
        if (s_cnt[3]) atomicAdd(&A.counters[6], (unsigned long long)s_cnt[3]);
        if (s_cnt[5]) atomicAdd(&A.counters[13], (unsigned long long)s_cnt[5]);
        if (s_cnt[4] > (unsigned)A.counters[12]) atomicMax(&A.counters[12], (unsigned long long)s_cnt[4]);   // longest trace since b200_run_sims began
    }
    __syncthreads();
    if (out.ask) {
        int pos = s_wreq[TPB / 32] + __popc(askmask & ((1u << (threadIdx.x & 31)) - 1u));
        for (int i = 0; i < (int)(threadIdx.x >> 5); ++i) pos += s_wreq[i];
        A.req[pos] = make_uint2((uint32_t)g, (uint32_t)out.my_o | ((uint32_t)gp.lane << 28));
    }
}

// continue the expansions that had to wait for k_gc (children resume_a..6), then queue their evaluations
__global__ void __launch_bounds__(TPB) k_expand_resume(Arena A) {
    __shared__ __align__(16) uint32_t s_stage[GROUPS_PER_BLOCK * STAGE_GROUP_WORDS];
    Grp gp;
    const int item = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 3);       // the games this step's k_select_expand queued for k_gc
    if (item >= A.n_req[1]) return;
    const int g = A.gc_list[item];
    if (A.pending[g] != PEND_EXPAND) return;
    gp.sync();
    if (gp.lane == 0) A.pending[g] = PEND_NONE;
    int status = A.status[g];
    if (status != ST_OK) return;                         // k_gc found the arena full: the reference dies here
    int D = A.trace_len[g];
    int leaf = A.trace[(size_t)g * A.trace_max + D - 1];
    uint32_t w[REC_WORDS];
    load_rec(A.rec + node_at(A, g, leaf) * REC_WORDS, w);
    int c, o, a_stop; float s;
    expand_leaf(A, gp, g, leaf, w, c, o, s, status, A.resume_a[g], false, a_stop, s_stage + (threadIdx.x >> 3) * STAGE_GROUP_WORDS, nullptr);
    if (status == ST_OK) {
        ArenaAcc acc(A, g);
        acc.children(leaf, gp.lane, c, o, s);            // children 0..resume_a-1 were linked before the collection
        Uniq u = finish_expansion(A, gp, g, leaf, c, o, s);
        if (A.mode == MODE_LP) request_lp_evals(A, gp, g, u, o);
        if (gp.lane == 0) A.leaf_kind[g] = LEAF_EXPANDED;
    } else if (gp.lane == 0) {
        A.status[g] = status;
    }
}

// ---------------------------------------------------------------- remove_nodes (agent.py:187-257), one CTA per game
// get_all_childs (core.h:32-50) as a level-synchronous parallel BFS, update_available (agent.py:187-204) as ordered
// compaction (ascending free lists, popped from the back), reset_arrays (agent.py:227-244) including its pop-by-stale-game
// behaviour (see stale_pop), then both hash tables are rebuilt from their surviving entries.
constexpr int GC_THREADS = 256;

__device__ __forceinline__ bool test_and_set_mark(uint8_t *mark, int i) {
    unsigned *wp = reinterpret_cast<unsigned *>(mark + (i & ~3));
    unsigned bit = 1u << (8 * (i & 3));
    return (atomicOr(wp, bit) & bit) == 0u;
}

__device__ __forceinline__ int block_excl_scan(int flag, int *s_warp, int &total) {   // 256 threads; returns rank of this thread
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned m = __ballot_sync(0xffffffffu, flag);
    int rank = __popc(m & ((1u << lane) - 1u));
    __syncthreads();
    if (lane == 0) s_warp[wid] = __popc(m);
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < GC_THREADS / 32; ++i) { int v = s_warp[i]; if (i < wid) off += v; tot += v; }
    total = tot;
    return off + rank;
}

__global__ void __launch_bounds__(GC_THREADS) k_gc(Arena A) {
    __shared__ int s_n[2];
    __shared__ int s_warp[GC_THREADS / 32];
    const int n_items = A.n_req[1];
    const int t = threadIdx.x;
    const int M = A.M, H = A.H;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int g = A.gc_list[item];
        if (A.pc && t == 0) A.pc_len[g] = 0;       // path cache: a collection (or the tree drop that may follow it) invalidates it
        uint8_t *nmark = A.nmark + (size_t)blockIdx.x * M, *omark = A.omark + (size_t)blockIdx.x * M;   // scratch of this CTA (a pool of gridDim.x sets,
        int32_t *q0 = A.gc_queue + (size_t)blockIdx.x * 2 * M, *q1 = q0 + M;                            // not one per game: 10 bytes per slot saved)
        int32_t *rowb = A.row + (size_t)g * M * ROW_WORDS;
        uint2 *ntab = A.ntab + (size_t)g * H, *otab = A.otab + (size_t)g * H;
        const uint32_t *recb = A.rec + (size_t)g * M * REC_WORDS;
        const int root = A.root[g];
        __syncthreads();
        for (int i = t; i < M / 4; i += GC_THREADS) { reinterpret_cast<unsigned *>(nmark)[i] = 0u; reinterpret_cast<unsigned *>(omark)[i] = 0u; }
        for (int i = (M / 4) * 4 + t; i < M; i += GC_THREADS) { nmark[i] = 0; omark[i] = 0; }
        __syncthreads();
        if (t == 0) {                                        // core.h:32-50: the null node 0 is always traversed
            nmark[0] = 1;
            int n = 0;
            if (root != 0) { nmark[root] = 1; q0[n++] = root; }
            s_n[0] = n; s_n[1] = 0;
        }
        __syncthreads();
        int32_t *cur = q0, *nxt = q1;
        for (;;) {
            const int nc = s_n[0];
            if (nc == 0) break;
            for (int i = t; i < nc * 7; i += GC_THREADS) {
                int c = rowb[(size_t)cur[i / 7] * ROW_WORDS + (i % 7)];
                if (c != 0 && test_and_set_mark(nmark, c)) nxt[atomicAdd(&s_n[1], 1)] = c;
            }
            __syncthreads();
            if (t == 0) { s_n[0] = s_n[1]; s_n[1] = 0; }
            int32_t *tmp = cur; cur = nxt; nxt = tmp;
            __syncthreads();
        }
        // observations of occupied nodes stay (agent.py:198); n_to_o[i] lives in o[7]
        for (int i = t; i < M; i += GC_THREADS)
            if (nmark[i]) omark[rowb[(size_t)i * ROW_WORDS + 15]] = 1;
        __syncthreads();
        // ascending complements (agent.py:192,201)
        int32_t *nfree = A.nfree + (size_t)g * M, *ofree = A.ofree + (size_t)g * M;
        int nn = 0, no = 0;
        for (int base = 0; base < M; base += GC_THREADS) {
            int i = base + t, tot;
            int fn = i < M && !nmark[i], fo = i < M && !omark[i];
            int r = block_excl_scan(fn, s_warp, tot);
            if (fn) nfree[nn + r] = i;
            nn += tot;
            r = block_excl_scan(fo, s_warp, tot);
            if (fo) ofree[no + r] = i;
            no += tot;
        }
        __syncthreads();
        // reset_arrays: node table.  stale_pop: erase BY THE FREED SLOT'S CURRENT GAME (agent.py:229-232); a slot freed
        // at an earlier collection still holds its old state, which may equal a live node's: that node loses its entry.
        if (A.stale_pop) {
            for (int j = t; j < nn; j += GC_THREADS) {
                const uint4 *mine = reinterpret_cast<const uint4 *>(recb + (size_t)nfree[j] * REC_WORDS);
                uint4 m0 = mine[0], m1 = mine[1], m2 = mine[2], m3 = mine[3], m4 = mine[4];
                uint32_t w[REC_WORDS] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w, m2.x, m2.y, m2.z, m2.w,
                                         m3.x, m3.y, m3.z, m3.w, m4.x, m4.y, m4.z, m4.w};
                uint32_t h = fold32(hash_words(w, REC_WORDS));
                uint32_t p = tab_home(h, H);
                for (;;) {
                    uint2 e = ntab[p];
                    if (e.y == 0u) break;
                    if (e.y != 0xffffffffu && e.x == h) {
                        const uint4 *c = reinterpret_cast<const uint4 *>(recb + (size_t)e.y * REC_WORDS);
                        uint4 c0 = c[0], c1 = c[1], c2 = c[2], c3 = c[3], c4 = c[4];
                        bool eq = c0.x == m0.x && c0.y == m0.y && c0.z == m0.z && c0.w == m0.w && c1.x == m1.x && c1.y == m1.y &&
                                  c1.z == m1.z && c1.w == m1.w && c2.x == m2.x && c2.y == m2.y && c2.z == m2.z && c2.w == m2.w &&
                                  c3.x == m3.x && c3.y == m3.y && c3.z == m3.z && c3.w == m3.w && c4.x == m4.x && c4.y == m4.y &&
                                  c4.z == m4.z && c4.w == m4.w;
                        if (eq) { ntab[p].y = 0xffffffffu; break; }
                    }
                    p = tab_next(p, H);
                }
            }
        } else {
            for (int p = t; p < H; p += GC_THREADS) { uint32_t y = ntab[p].y; if (y != 0u && y != 0xffffffffu && !nmark[y]) ntab[p].y = 0xffffffffu; }
        }
        for (int p = t; p < H; p += GC_THREADS) { uint32_t y = otab[p].y; if (y != 0u && y != 0xffffffffu && !omark[y]) otab[p].y = 0xffffffffu; }
        __syncthreads();
        // rebuild both tables from their surviving entries (the BFS queues are free again: 2M ints = M pairs)
        for (int tb = 0; tb < 2; ++tb) {
            uint2 *tab = tb ? otab : ntab;
            uint2 *list = reinterpret_cast<uint2 *>(q0);
            if (t == 0) s_n[0] = 0;
            __syncthreads();
            for (int p = t; p < H; p += GC_THREADS) {
                uint2 e = tab[p];
                if (e.y != 0u && e.y != 0xffffffffu) list[atomicAdd(&s_n[0], 1)] = e;
                tab[p] = make_uint2(0u, 0u);
            }
            __syncthreads();
            const int cnt = s_n[0];
            for (int j = t; j < cnt; j += GC_THREADS) {      // keys are unique, so the claim order is free
                uint2 e = list[j];
                uint32_t p = tab_home(e.x, H);
                while (atomicCAS(&tab[p].y, 0u, e.y) != 0u) p = tab_next(p, H);
                tab[p].x = e.x;
            }
            __syncthreads();
        }
        // zero the freed rows (agent.py:234-235; node_to_obs is not in self.arrays: o[7] stays), statistics and keys
        constexpr int RQ = ROW_WORDS / 4;
        for (int i = t; i < nn * RQ; i += GC_THREADS) {
            int4 *r = reinterpret_cast<int4 *>(rowb + (size_t)nfree[i / RQ] * ROW_WORDS) + (i % RQ);
            *r = make_int4(0, 0, 0, (i % RQ) == 3 ? r->w : 0);
        }
        if (A.nstat) {
            float *nsb = A.nstat + (size_t)g * M * NSTAT_WORDS, *ndb = A.ndist + (size_t)g * M * A.dist_bins;
            for (int i = t; i < nn * NSTAT_WORDS; i += GC_THREADS) nsb[(size_t)nfree[i / NSTAT_WORDS] * NSTAT_WORDS + (i % NSTAT_WORDS)] = 0.f;
            for (int i = t; i < nn * A.dist_bins; i += GC_THREADS) ndb[(size_t)nfree[i / A.dist_bins] * A.dist_bins + (i % A.dist_bins)] = 0.f;
        }
        int4 *statb = A.stat + (size_t)g * M;
        uint4 *keyb = reinterpret_cast<uint4 *>(A.key + (size_t)g * M * KEY_WORDS);
        // store_nodes (agents/ValueSim.py:122-159, agent.cpp:777-819): freed observations with visit >= min_visits_to_store and not
        // `end` go to the replay memory before their statistics are zeroed; storing stops when the memory is full (ValueSim.py:152-154)
        if (A.replay) {
            // in ascending index order like the reference's loop (rows of one collection are contiguous and ordered; the memory stops
            // taking rows when it is full: `if(++memory_index == memory_size) break;`, agent.cpp:817 / ValueSim.py:152-154)
            for (int base = 0; base < no; base += GC_THREADS) {
                const int i = base + t;
                int o = 0; int4 st = make_int4(0, 0, 0, 0);
                bool keep = false;
                if (i < no) {
                    o = ofree[i];
                    st = statb[o];
                    keep = !(st.x < A.replay_min_visits || st.x == 0 || st.w != 0);
                }
                int tot;
                const int r = block_excl_scan(keep ? 1 : 0, s_warp, tot);
                if (t == 0) s_n[0] = tot ? atomicAdd(A.replay_count, tot) : 0;
                __syncthreads();
                const int slot = s_n[0] + r;
                if (keep && slot < A.replay_cap) {
                    uint8_t *dst = A.replay + (size_t)slot * 212;
                    const uint32_t *k = A.key + ((size_t)g * M + o) * KEY_WORDS;
                    for (int rr = 0; rr < 20; ++rr) {
                        const uint32_t row = (k[rr >> 1] >> ((rr & 1) * 16)) & 0x3ffu;
                        for (int c = 0; c < 10; ++c) dst[rr * 10 + c] = (uint8_t)((row >> c) & 1u);
                    }
                    for (int j = 0; j < 4; ++j) dst[(k[10] >> (8 * j)) & 0xffu] = 0xff;            // int8 -1: the falling piece
                    const float f[3] = {__int_as_float(st.y), __int_as_float(st.z), (float)st.x};
                    memcpy(dst + 200, f, 12);
                }
                __syncthreads();
            }
            if (t == 0 && *A.replay_count > A.replay_cap) atomicMin(A.replay_count, A.replay_cap);   // rows past the capacity were not stored
            __syncthreads();
        }
        for (int i = t; i < no; i += GC_THREADS) statb[ofree[i]] = make_int4(0, 0, 0, 0);
        for (int i = t; i < no * 3; i += GC_THREADS) keyb[(size_t)ofree[i / 3] * 3 + (i % 3)] = make_uint4(0, 0, 0, 0);
        if (t == 0) {
            A.n_nfree[g] = nn; A.n_ofree[g] = no;
            atomicAdd(&A.counters[3], 1ull);
            if (nn == 0) A.status[g] = ST_ARENA_FULL;        // reference: IndexError at agent.py:99 / UB at agent.cpp:227-231
        }
        // overflow_reset policy (beyond the reference, bench only): a collection that recovers fewer than gc_min_gain slots means the
        // reachable set itself fills the arena; the reference would collect again at almost every expansion from here on (a
        // whole-arena sweep for a handful of slots) and then die.  The tree is dropped here, by the whole block, and the next
        // k_select_expand / k_update_root only re-roots it (ST_RESET_DONE).
        if (A.overflow_reset && nn < A.gc_min_gain) {
            __syncthreads();
            int4 *rows = reinterpret_cast<int4 *>(rowb);
            for (int i = t; i < M * (ROW_WORDS / 4); i += GC_THREADS) rows[i] = make_int4(0, 0, 0, 0);
            for (int i = t; i < M; i += GC_THREADS) statb[i] = make_int4(0, 0, 0, 0);
            for (int i = t; i < M * 3; i += GC_THREADS) keyb[i] = make_uint4(0, 0, 0, 0);
            for (int i = t; i < H; i += GC_THREADS) { ntab[i] = make_uint2(0, 0); otab[i] = make_uint2(0, 0); }
            if (A.nstat) {
                float *nsb = A.nstat + (size_t)g * M * NSTAT_WORDS, *ndb = A.ndist + (size_t)g * M * A.dist_bins;
                for (int i = t; i < M * NSTAT_WORDS; i += GC_THREADS) nsb[i] = 0.f;
                for (size_t i = t; i < (size_t)M * A.dist_bins; i += GC_THREADS) ndb[i] = 0.f;
            }
            for (int i = t; i < M - 1; i += GC_THREADS) { nfree[i] = i + 1; ofree[i] = i + 1; }
            if (t == 0) {
                A.n_nfree[g] = M - 1; A.n_ofree[g] = M - 1;
                A.status[g] = ST_RESET_DONE;
                atomicAdd(&A.counters[7], 1ull);
            }
        }
        __syncthreads();
    }
}

// remove_nodes() called by the driver (TreeAgent.remove_nodes is a public method, agents/agent.py:246-257): queue every game whose
// free list is shorter than min_free for ONE batched k_gc launch (all SMs busy), instead of one nearly empty k_gc launch per
// simulation step in which some game happens to run dry (a single collection is a ~1 ms latency chain the whole step waits for).
__global__ void k_gc_request(Arena A, int min_free) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= A.G || A.status[g] != ST_OK || A.pending[g] != PEND_NONE) return;
    if (A.n_nfree[g] < min_free) A.gc_list[atomicAdd(A.n_req + 1, 1)] = g;
}

// ---------------------------------------------------------------- test evaluator (shared definition with oracle/mcts_oracle.c)
__device__ __forceinline__ void synthetic_eval(const uint32_t *k, float &v, float &var) {
    uint32_t h = 2166136261u;
#pragma unroll
    for (int i = 0; i < 11; ++i) { h ^= k[i]; h *= 16777619u; }
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    v = (float)((h >> 7) & 0x3fffu) * 0.00390625f;
    var = 0.5f + (float)((h >> 21) & 0x3ffu) * 0.0625f;
}

__global__ void k_eval_synthetic(Arena A) {
    int n = *A.n_req;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 r = A.req[i];
        int g = (int)r.x, o = (int)(r.y & 0x0fffffffu), slot = (int)(r.y >> 28);
        float v, var;
        synthetic_eval(A.key + node_at(A, g, o) * KEY_WORDS, v, var);
        A.eval_out[(size_t)g * 8 + slot] = make_float2(v, var);
    }
}

// ---------------------------------------------------------------- random rollout (Vanilla.py:47-55), one thread per game
__global__ void k_rollout(Arena A) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= A.G || A.status[g] != ST_OK || A.leaf_kind[g] != LEAF_EXPANDED) return;
    int leaf = A.trace[(size_t)g * A.trace_max + A.trace_len[g] - 1];
    uint32_t w[REC_WORDS];
    load_rec(A.rec + node_at(A, g, leaf) * REC_WORDS, w);
    Game gm;
    unpack(gm, w);
    uint32_t sr = A.srng[g];
    unsigned steps = 0;
    while (!gm.end) { play(gm, (int)(rng_next(sr) % 7u)); ++steps; }
    A.srng[g] = sr;
    A.rollout_val[g] = (float)gm.score;
    atomicAdd(&A.counters[5], (unsigned long long)steps);
}

// ---------------------------------------------------------------- backup (core.h:226-381)
// The reference walks the trace leaf -> root with two dependent gathers per level.  Here the 32 lanes of a warp fetch 32
// levels at once (node meta, then statistics), the Welford recurrence then runs in exactly the reference's order (same
// welford_level code, v carried in double), and the statistics are written back in parallel.  If an observation
// occurs twice among the levels in flight (statistics are shared between nodes, agent.py:116-128) the lanes fall back
// to the scalar walk.  Everything the backup never writes (trace, row fields, evaluator outputs) is loaded as early as
// possible: the first window's node fields together with the leaf's child row, the next window's while the current one
// is folded, so that only the statistics loads sit on the dependent chain (a DRAM access is ~2.4 k clk here).
// One warp per game (k_backup); leaf_kind[g] is set to LEAF_DONE once the trace is folded, so a second backup of the same
// trace does nothing.
__device__ __forceinline__ void backup_game(const Arena &A, int g, int lane, unsigned *bitmap) {
    constexpr unsigned mask = 0xffffffffu;
    ArenaAcc acc(A, g);
    const int D = A.trace_len[g];
    const int kind = A.leaf_kind[g];
    if (kind == LEAF_SUSPENDED || kind == LEAF_DONE || D <= 0) return;
    // path cache (search_dev.cuh): pcl = the entries the walk left valid (0: off, or invalidated by a collection since); `stale` = this lane's
    // shallowest level whose entry holds an out-of-date copy after this backup (min-reduced at the end)
    const int pcl = (bitmap && acc.pcg) ? A.pc_len[g] : 0;
    int stale = pcl;
    // ---- early loads: trace entries of the first window, then their node fields + the leaf's child row + evaluator outputs
    const int n0 = D < 32 ? D : 32;
    int tidx = 0;
    if (lane == 0) tidx = acc.get_trace(D - 1);
    const bool lp_children = A.mode == MODE_LP && kind == LEAF_EXPANDED;
    int wo = -1 - lane; float wsc = 0.f;                      // this lane's level of the current window: observation (| the walk's pick << 28), score
    if (lane < n0) acc.get_trace_meta_raw(D - 1 - lane, wo, wsc); // recorded by the walk: one coalesced read instead of a gather per level
    const int leaf = __shfl_sync(mask, tidx, 0);
    int c = 0, o = 0; float s = 0.f;
    float2 ev = make_float2(0.f, 0.f);
    if (lp_children && lane < 8) { acc.children(leaf, lane, c, o, s); ev = A.eval_out[(size_t)g * 8 + lane]; }
    const float leaf_score = __shfl_sync(mask, wsc, 0);
    double v = (double)leaf_score, var = 0.0;
    if (A.mode == MODE_LP) {
        if (kind == LEAF_EXPANDED) {
            // core.h:340-366: initialise unvisited unique children, then average score + gamma*value and the variances
            Grp gp;                                   // lanes 0-7 form the group that holds the 7 child slots
            double v_tmp = 0.0, var_tmp = 0.0;
            int k = 0;
            if (lane < 8) {
                Uniq u = unique_children(gp, c, o, s);
                int4 st = make_int4(0, 0, 0, 0);
                if (u.is_first) {
                    st = acc.stat(o);
                    if (st.x == 0) {                                           // core.h:344-353
                        bool cend = A.lp_end_from_obs ? (st.w != 0) : false;   // SURVEY N1
                        st.x = 1; st.y = __float_as_int(cend ? 0.f : ev.x); st.z = __float_as_int(cend ? 0.f : ev.y);
                        acc.set_stat(o, st);
                    }
                }
                k = __popc(u.first_mask);
#pragma unroll
                for (int j = 0; j < 7; ++j) {                                  // list order = slot order of first occurrences
                    float sj = gp.bcast(u.rep_s, j), valj = gp.bcast(__int_as_float(st.y), j), s2j = gp.bcast(__int_as_float(st.z), j);
                    if ((u.first_mask >> j) & 1u) {
                        v_tmp = __dadd_rn(v_tmp, __dadd_rn((double)sj, __dmul_rn(A.gamma, (double)valj)));   // core.h:355
                        var_tmp = __dadd_rn(var_tmp, (double)s2j);
                    }
                }
            }
            k = __shfl_sync(mask, k, 0);
            v_tmp = __shfl_sync(mask, v_tmp, 0);
            var_tmp = __shfl_sync(mask, var_tmp, 0);
            v = __ddiv_rn(v_tmp, (double)k);                                   // core.h:364
            if (A.lp_var_gamma2) var = __dmul_rn(var_tmp, __ddiv_rn(__dmul_rn(A.gamma, A.gamma), (double)k));   // core.h:365
            else { var = __ddiv_rn(var_tmp, (double)k); v = (double)(float)v; var = (double)(float)var; }        // agent.cpp:557-562
            __syncwarp(mask);
        }
    } else if (A.mode == MODE_SINGLE) {
        if (kind == LEAF_EXPANDED) {
            float2 e = A.eval_out[(size_t)g * 8 + 7];
            v = (double)__fadd_rn(leaf_score, e.x);      // ValueSim.py:86 int + np.float32 -> float32 (numpy >= 2)
            var = (double)e.y;
        }
    } else if (kind == LEAF_EXPANDED) {
        v = (double)A.rollout_val[g]; var = A.rollout_variance;                // Vanilla.py:53-54
    }
    // ---- core.h:244-259 along the trace, 32 levels per round
    for (int top = D - 1; top >= 0; top -= 32) {
        const int n = top + 1 < 32 ? top + 1 : 32;      // levels top, top-1, ..., top-n+1 -> lanes 0..n-1
        const int oraw = wo;
        const int o = oraw < 0 ? oraw : (oraw & (int)TMETA_OBS_MASK); const float sc = wsc;
        int4 st = make_int4(0, 0, 0, 0);
        const bool dup = __popc(__match_any_sync(mask, o)) > 1;
        const bool any_dup = __any_sync(mask, dup);
        if (!any_dup && lane < n) st = acc.stat(o, top - lane);
        {   // the next window's node fields, in flight while this window is folded
            const int ntop = top - 32;
            wo = -1 - lane; wsc = 0.f;
            if (ntop >= 0 && lane <= ntop) acc.get_trace_meta_raw(ntop - lane, wo, wsc);
        }
        // path cache: a bitmap of the trace's own observations for the staleness scan below; a bit already set by a DEEPER window = the same
        // observation twice on the trace: the deeper occurrence's own record holds an intermediate value
        if (pcl > 0) {
            if (lane < n) {
                const unsigned bit = 1u << (o & 31);
                const unsigned old = atomicOr(&bitmap[o >> 5], bit);
                if ((old & bit) && top - lane < stale) stale = top - lane;
            }
            if (any_dup && top - n < stale) stale = top - n < 0 ? 0 : top - n;   // the same inside this window: no own records are written for it
        }
        if (any_dup) {                                  // shared observation inside the window: scalar walk for this window
            if (lane == 0) {
                for (int i = top; i > top - n; --i) {
                    int oo; float ss;
                    acc.get_trace_meta(i, oo, ss);
                    int4 s2 = acc.stat(oo);
                    welford_level(s2, v, var, ss, A.gamma);
                    acc.set_stat(oo, s2);
                }
            }
            v = __shfl_sync(mask, v, 0);
            __syncwarp(mask);
            continue;
        }
        // The value chain v <- gamma*(v - score) + score (core.h:244,259) does not depend on the statistics: every lane
        // walks it (three dependent double operations per level) and keeps the value entering its own level; the expensive
        // Welford updates (core.h:245-258) of the whole window then run in parallel, one level per lane.
        double vin = v;
        for (int j = 0; j < n; ++j) {
            const double scj = (double)__shfl_sync(mask, sc, j);
            if (lane == j) vin = v;
            v = __dadd_rn(__dmul_rn(A.gamma, __dsub_rn(v, scj)), scj);
        }
        if (lane < n) {
            welford_level(st, vin, var, sc, A.gamma); acc.set_stat(o, st, top - lane);
            if (pcl > 0) acc.pown[top - lane] = make_int4(st.x, st.y, st.z, 0);   // the level's own record: what the walk one level up reads for its picked child
        }
        __syncwarp(mask);
    }
    if (pcl > 0) {
        // ---- staleness scan: a cached child observation that is some trace node's own WITHOUT being its level's picked child (the same
        // observation under two nodes of the path: statistics are shared between nodes, agent.py:116-128) still holds its fill-time value.
        // One level per lane: eight u16 of pc_sib (seven child observations, 0 = not a slot the walk reads; the picked slot).
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) stale = min(stale, __shfl_xor_sync(mask, stale, d));
        const int upto = stale;                         // entries at or beyond a stale level are dropped anyway
        int stale2 = upto;
        const uint4 *sib = reinterpret_cast<const uint4 *>(acc.psib);
        for (int L = lane; L < upto; L += 32) {
            const uint4 sv = sib[L];
            const unsigned wv[4] = {sv.x, sv.y, sv.z, sv.w};
            const int pk = (int)(sv.w >> 16);
            bool hit = false;
#pragma unroll
            for (int a = 0; a < 7; ++a) {
                const unsigned oc = (wv[a >> 1] >> ((a & 1) * 16)) & 0xffffu;
                hit |= oc != 0u && a != pk && ((bitmap[oc >> 5] >> (oc & 31)) & 1u);
            }
            if (hit) { stale2 = L; break; }             // this lane's levels ascend: the first hit is its shallowest
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) stale2 = min(stale2, __shfl_xor_sync(mask, stale2, d));
        if (lane == 0 && stale2 < pcl) A.pc_len[g] = stale2;
    }
    if (lane == 0) A.leaf_kind[g] = LEAF_DONE;
    __syncwarp(mask);
}

constexpr int BACKUP_MINB = 9;   // resident 128-thread blocks per SM the register budget is cut for (9 = what 56 registers give)
// Dynamic shared memory: with the path cache on, one bitmap of max_nodes bits per warp (the observations of the game's trace), else none.
__global__ void __launch_bounds__(128, BACKUP_MINB) k_backup(Arena A, int bitmap_words) {
    extern __shared__ unsigned s_bitmap[];
    const int g = blockIdx.x * 4 + (threadIdx.x >> 5);
    unsigned *bm = bitmap_words ? s_bitmap + (threadIdx.x >> 5) * bitmap_words : nullptr;
    for (int i = threadIdx.x & 31; i < bitmap_words; i += 32) bm[i] = 0u;
    __syncwarp();
    if (g >= A.G || A.status[g] != ST_OK) return;
    backup_game(A, g, threadIdx.x & 31, bm);
}

// ---------------------------------------------------------------- distributional mode (config 5): evaluator + backup
// test evaluator, shared definition with oracle/mcts_oracle.c: mo_synthetic_dist
__global__ void k_eval_synthetic_dist(Arena A) {
    int n = *A.n_req;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 r = A.req[i];
        int g = (int)r.x, o = (int)(r.y & 0x0fffffffu);
        const uint32_t *k = A.key + node_at(A, g, o) * KEY_WORDS;
        uint32_t sum = 0;
        float *out = A.dist_eval + (size_t)g * A.dist_bins;
        for (int pass = 0; pass < 2; ++pass)
            for (int b = 0; b < A.dist_bins; ++b) {
                uint32_t h = 2166136261u;
                for (int j = 0; j < 11; ++j) { h ^= k[j]; h *= 16777619u; }
                h ^= (uint32_t)b * 0x9E3779B9u; h *= 16777619u;
                h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
                uint32_t raw = ((h >> 9) & 0xffu) + 1u;
                if (pass == 0) sum += raw; else out[b] = __fdiv_rn((float)raw, (float)sum);
            }
    }
}

// backup_trace_distributional (core_distributional.py:109-124), one warp per game, lanes over the histogram bins.
// The trace levels are independent of each other (dist and r are fixed), so each level is: shift the evaluator's
// histogram by (r - reward[idx]) (closed-form gather of shift_distribution, same add order per bin; the clamped top bin is
// summed sequentially), fold it into the node's running average, update the node's Welford statistics.
__global__ void __launch_bounds__(128) k_dist_backup(Arena A) {
    __shared__ float s_dist[4][64];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * 4 + wid;
    if (g >= A.G || A.status[g] != ST_OK) return;
    const int D = A.trace_len[g], kind = A.leaf_kind[g];
    if (kind == LEAF_SUSPENDED || D <= 0) return;
    const int bins = A.dist_bins, T = bins - 1;
    const int32_t *trace = A.trace + (size_t)g * A.trace_max;
    const int leaf = trace[D - 1];
    float *nsb = A.nstat + (size_t)g * A.M * NSTAT_WORDS, *ndb = A.ndist + (size_t)g * A.M * bins;
    const double r = (double)__int_as_float(A.row[node_at(A, g, leaf) * ROW_WORDS + 23]);   // leaf_game.getScore(), DistValueSimOnline.py:64
    float *d = s_dist[wid];
    for (int b = lane; b < bins; b += 32)
        d[b] = kind == LEAF_EXPANDED ? A.dist_eval[(size_t)g * bins + b] : (b == 0 ? 1.f : 0.f);   // v_dummy, DistValueSimOnline.py:26-27
    __syncwarp();
    const double delta = (A.dist_vmax - A.dist_vmin) / bins;
    double mean = 0.0;                                               // mean_dist, core_distributional.py:39-45 (sequential order)
    for (int b = 0; b < bins; ++b) mean = __dadd_rn(mean, __dmul_rn((double)d[b], (b + 0.5) * delta));
    for (int t = 0; t < D; ++t) {
        const int idx = trace[t];
        float *ns = nsb + (size_t)idx * NSTAT_WORDS, *nd = ndb + (size_t)idx * bins;
        const float ns0 = ns[0], ns1 = ns[1], ns2 = ns[2], ns4 = ns[4];
        const double _r = r - (double)ns2;
        const double bin_shift = _r / delta, frac = bin_shift - floor(bin_shift);
        const int s = (int)bin_shift;                                // (int)(b + bin_shift) = b + s for bin_shift >= 0
        for (int tb = lane; tb < bins; tb += 32) {
            float acc = 0.f;
            if (tb < T) {
                int b1 = tb - s - 1, b2 = tb - s;
                if (b1 >= 0 && b1 < bins) acc = (float)__dadd_rn((double)acc, __dmul_rn((double)d[b1], frac));          // its upper target
                if (b2 >= 0 && b2 < bins) acc = (float)__dadd_rn((double)acc, __dmul_rn((double)d[b2], 1.0 - frac));    // its lower target
            } else {
                int b0 = T - s - 1;
                if (b0 >= 0 && b0 < bins) acc = (float)__dadd_rn((double)acc, __dmul_rn((double)d[b0], frac));
                for (int b = (T - s < 0 ? 0 : T - s); b < bins; ++b) {                                                   // clamped bins
                    acc = (float)__dadd_rn((double)acc, __dmul_rn((double)d[b], 1.0 - frac));
                    acc = (float)__dadd_rn((double)acc, __dmul_rn((double)d[b], frac));
                }
            }
            float num = __fadd_rn(__fmul_rn(nd[tb], ns0), acc);
            nd[tb] = (float)((double)num / ((double)ns0 + 1.0));
        }
        if (lane == 0) {
            const double x = mean + _r;
            const float n1 = __fadd_rn(ns0, 1.f);
            const double dl = x - (double)ns1;
            const float m1 = (float)((double)ns1 + dl / (double)n1);
            const double dl2 = x - (double)m1;
            const float m2 = (float)((double)ns4 + dl * dl2);
            ns[0] = n1; ns[1] = m1; ns[4] = m2;
            if (n1 > 1.f) ns[3] = (float)((double)m2 / ((double)n1 - 1.0));
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- compute_stats / get_action (agent.py:153-185)
__global__ void k_root_stats(Arena A, float *stats, int32_t *action) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= A.G) return;
    ArenaAcc acc(A, g);
    int root = A.root[g];
    int ro; float rs;
    acc.meta(root, ro, rs);
    float best = 0.f; int arg = 0;
    if (A.mode == MODE_DIST) {      // DistValueSimOnline.py:77-104: visit, mean + reward - root reward, variance; argmax of row 1
        const float *nsb = A.nstat + (size_t)g * A.M * NSTAT_WORDS;
        const float rr = nsb[(size_t)root * NSTAT_WORDS + 2];
        for (int a = 0; a < 7; ++a) {
            int c = A.row[node_at(A, g, root) * ROW_WORDS + a];
            const float *ns = nsb + (size_t)c * NSTAT_WORDS;
            float val = __fsub_rn(__fadd_rn(ns[1], ns[2]), rr);
            stats[(size_t)g * 21 + a] = ns[0]; stats[(size_t)g * 21 + 7 + a] = val; stats[(size_t)g * 21 + 14 + a] = ns[3];
            if (a == 0 || val > best) { best = val; arg = a; }
        }
        action[g] = arg;
        return;
    }
    for (int a = 0; a < 7; ++a) {
        int c, o; float s;
        acc.children(root, a, c, o, s);
        int4 st = acc.stat(o);                                  // child 0 -> obs 0 -> zeros, as in the reference
        float diff = __fsub_rn(s, rs);                          // agent.py:171
        float val = __fadd_rn(__int_as_float(st.y), diff);      // agent.py:175
        stats[(size_t)g * 21 + a] = (float)st.x;
        stats[(size_t)g * 21 + 7 + a] = val;
        stats[(size_t)g * 21 + 14 + a] = __int_as_float(st.z);
        if (a == 0 || val > best) { best = val; arg = a; }      // np.argmax: first maximum
    }
    action[g] = arg;
}

// ---------------------------------------------------------------- single-call twins of core.cpp:20-26 (one group / one thread)
struct TwinArgs {
    const int32_t *child; int32_t *visit; float *value; float *variance; const float *score; const int32_t *n2o;
    int32_t *trace; uint32_t *rng; int32_t *out;
};

__global__ void k_twin_select(Arena A, TwinArgs t, int index, int low, int max_trace) {   // one warp; the first 8-lane group owns the tree
    RefAcc acc{t.child, t.visit, t.value, t.variance, t.score, t.n2o, t.trace, t.rng, &A};
    int D = 0, status = ST_OK;
    select_trace(acc, threadIdx.x < 8, index, low, max_trace, D, status);
    if (threadIdx.x == 0) { t.out[0] = D; t.out[1] = status; }
}

__global__ void k_twin_unique(Arena A, TwinArgs t, int index) {
    Grp gp;
    if (threadIdx.x >= 8) return;
    RefAcc acc{t.child, t.visit, t.value, t.variance, t.score, t.n2o, t.trace, t.rng, &A};
    int c, o; float s;
    acc.children(index, gp.lane, c, o, s);
    Uniq u = unique_children(gp, c, o, s);
    int pos = __popc(u.first_mask & ((1u << gp.lane) - 1u));
    if (u.is_first) { t.out[1 + pos] = u.rep_c; t.out[8 + pos] = o; }
    if (gp.lane == 0) t.out[0] = __popc(u.first_mask);
}

__global__ void k_twin_backup(Arena A, TwinArgs t, int D, double v, double var, double gamma, int mixture) {
    RefAcc acc{t.child, t.visit, t.value, t.variance, t.score, t.n2o, t.trace, t.rng, &A};
    if (mixture) backup_trace_mixture(acc, D, v, var, gamma);
    else backup_trace(acc, D, v, var, gamma);
}

__global__ void k_twin_backup_lp(Arena A, TwinArgs t, int D, const uint8_t *end, const int32_t *c_nodes, const int32_t *c_obs,
                                 int k, const float *v, const float *var, double gamma, int mixture, int averaged) {
    RefAcc acc{t.child, t.visit, t.value, t.variance, t.score, t.n2o, t.trace, t.rng, &A};
    int co[7]; float cs[7], ev[7], evar[7]; bool ce[7];
    for (int i = 0; i < k; ++i) { co[i] = c_obs[i]; cs[i] = t.score[c_nodes[i]]; ev[i] = v[i]; evar[i] = var[i]; ce[i] = end[c_nodes[i]] != 0; }
    float leaf_score = t.score[t.trace[D - 1]];
    lp_backup(acc, D, k, co, cs, ev, evar, ce, gamma, mixture != 0, averaged != 0, true, leaf_score);
}

// get_all_childs (core.h:32-50) on the reference layout: mark[] = 1 for every traversed index (0 included)
__global__ void k_twin_all_childs(const int32_t *child, int M, int index, uint8_t *mark, int32_t *queue) {
    if (threadIdx.x != 0) return;
    int head = 0, tail = 0;
    queue[tail++] = index; mark[index] = 1;
    while (head < tail) {
        int n = queue[head++];
        for (int a = 0; a < 7; ++a) {
            int c = child[(size_t)n * 7 + a];
            if (!mark[c]) { mark[c] = 1; queue[tail++] = c; }
        }
    }
}

}  // namespace b200
