// search_dev.cuh — device side of the per-move MCTS simulation loop (sm_100a).
//
// One 8-lane group (quarter warp) owns one game's tree for the whole kernel; lane a (0..6) is child slot /
// action a, lane 7 carries the node's own fields.  Trees never share memory between games, so there are no
// inter-game races and no atomics on tree state.
//
// Reference functions restated here (file:line in /root/reference):
//   get_unique_child_obs  agents/cppmodule/core.h:111-144        -> unique_children()
//   check_low             core.h:65-77                            -> inside select_trace()
//   policy_clt            core.h:83-105, special.h:26-33          -> clt_q(), select_trace()
//   select_trace_obs      core.h:167-224                          -> select_trace()
//   backup_trace_obs      core.h:226-260                          -> welford_level(), backup_trace()
//   backup_trace_obs_LP   core.h:303-381 (averaged, non-mixture)  -> lp_init_and_average()
//   new_node / expand     agents/agent.py:90-145                  -> new_node(), expand_leaf()
//   remove_nodes          agents/agent.py:187-257, core.h:32-50   -> collect_garbage()
//   compute_stats         agents/agent.py:153-185                 -> root_stats()
//
// Bit-exactness: every float/double operation that the reference evaluates (g++ -O3, x86-64, no FMA) is written
// with explicit round-to-nearest intrinsics so that nvcc cannot contract it into an FMA.
#pragma once
#include <stdint.h>
#include "tetris_dev.cuh"

namespace b200 {

constexpr int ROW_WORDS = 32;     // child row (one 128-byte line): c[8] | o[8] | s[8] | u[8]; u = the child list already de-duplicated (see link_word)
constexpr int ZTABLE_N = 65536;   // z(n) table computed on the host with the reference's libm (special.h:26-33)

enum : int { ST_OK = 0, ST_ARENA_FULL = 1, ST_TRACE_FULL = 2, ST_NEED_GC = 3, ST_RESET_DONE = 4 };   // RESET_DONE: k_gc dropped the tree (overflow_reset), only the re-rooting is left
enum : int { LEAF_TERMINAL = 0, LEAF_EXPANDED = 1, LEAF_SUSPENDED = 2, LEAF_DONE = 3 };   // DONE: the trace has been backed up
enum : int { PEND_NONE = 0, PEND_EXPAND = 1, PEND_ROOT = 2 };
enum : int { MODE_LP = 0, MODE_SINGLE = 1, MODE_VANILLA = 2, MODE_DIST = 3 };
constexpr int NSTAT_WORDS = 8;    // node_stats row: {visit, mean, reward, variance, M2, -, -, -} (agents/core_distributional.py:109-124)

// HBM layout (all arrays are [game][...]; SoA across games, records kept 16-byte aligned):
//   row      [G][M][24] i32/f32  node record: child ids c[0..6], c[7]=episode | child obs o[0..6], o[7]=own obs |
//                                 child scores s[0..6], s[7]=own score.  One 96-B read gives select everything that
//                                 the reference gathers from child[idx], n_to_o[c], score[c], score[idx].
//   stat     [G][M]     int4     observation statistics {visit, value, variance, end}  (one 128-bit load/store)
//   rec      [G][M][20] u32      packed game (SPEC §6), the node key
//   key      [G][M][12] u32      observation key (SPEC §6), the statistics key
//   ntab/otab[G][H]     uint2    open-addressing tables {hash32, index}, H = 1.5 M; index 0 empty, 0xffffffff deleted
//   nfree/ofree [G][M]  i32      free lists, popped from the back (agents/agent.py:72,99)
struct Arena {
    int G, M, H, trace_max;
    int mode, low, lp_end_from_obs, lp_var_gamma2, stale_pop, eval_kind, overflow_reset;
    int gc_min_gain;               // overflow_reset only: a collection that leaves fewer free slots than this drops the tree (see k_gc)
    double gamma, rollout_variance;
    int32_t *row; int4 *stat; uint32_t *rec; uint32_t *key;
    uint2 *ntab, *otab;
    int32_t *nfree, *ofree; int32_t *n_nfree, *n_ofree;
    int32_t *root, *episode, *status; uint32_t *srng;
    int32_t *trace, *trace_len, *leaf_kind;
    int2 *trace_meta;              // [G][trace_max] {own observation, own score bits} of every node on the trace, written by the walk (it has
                                   // both in lane 7 of the level it just loaded) so that the backup needs no second gather per level
    uint8_t *nmark, *omark; int32_t *gc_queue;
    // path cache (b200_set_path_cache; LP mode): for every level of the game's last trace the node, its row fields and the STATISTICS OF
    // ITS CHILDREN, so that the next walk, which retraces ~93 % of that path, reads sequential lines instead of chasing a row line and seven
    // statistics per level; pc_len[g] = how many leading levels are valid.  Layout: "path cache" below
    int4 *pc; int32_t *pc_var; int32_t *pc_len;
    uint4 *pc_sib; int4 *pc_own;   // [G][trace_max] per level: the children's observation ids (8 x u16, the last = the picked slot) | the level's OWN statistics
    uint32_t *cur;                 // [G][20] the live game of each tree (the object play.py owns)
    const float *ztable;
    uint2 *req; int32_t *n_req;    // evaluation requests {game, obs | slot<<28}; n_req[0] = count, n_req[1] = games queued for k_gc
    int32_t *gc_list, *pending, *resume_a;   // [G] games waiting for a collection, what to resume, and at which child
    // replay memory (ValueSim.memory, agents/ValueSim.py:25-30; agent.cpp:610-613): 212-byte rows {int8 state[200], f32 value,
    // f32 variance, f32 visit}, filled by k_gc from the observations a collection frees (ValueSim.py:101-159)
    uint8_t *replay; int32_t *replay_count; int replay_cap, replay_min_visits;
    // finished episodes of the last update_root(auto_reset) calls: {game, score, line_clears, episode} per finished game, what play.py:161-177
    // prints as its `Episode: .. Score: .. Lines Cleared: ..` line before it resets the game; drained by b200_finished_games
    int32_t *fin_log; int32_t *fin_count; int fin_cap;
    float2 *eval_out;              // [G][8] (value, variance) per child slot; slot 7 = the leaf itself
    float *rollout_val;            // [G]
    // distributional mode (agents/core_distributional.py; BASELINE config 5): node-indexed statistics and value histograms
    float *nstat; float *ndist; float *dist_eval; int dist_bins; double dist_vmin, dist_vmax;   // [G][M][8], [G][M][bins], [G][bins]
    unsigned long long *counters;  // [8] 0 sims 1 expansions 2 eval requests 3 gcs 4 trace levels 5 rollout steps 6 new nodes
    unsigned long long *prof;      // timing mode only: clock64 sums of k_select_expand {select, leaf load, expand, finish, groups sampled}
};

// ------------------------------------------------------------------ group helpers
struct Grp {
    unsigned mask; int lane;   // lane within the 8-lane group
    __device__ __forceinline__ Grp() {
        int l = threadIdx.x & 31;
        lane = l & 7;
        mask = 0xffu << (l & 24);
    }
    template <typename T> __device__ __forceinline__ T bcast(T v, int src) const { return __shfl_sync(mask, v, src, 8); }
    __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(mask, p) >> ((threadIdx.x & 31) & 24)) & 0xffu; }
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
};

// The same interface with the CONSTANT full mask: legal only where all 32 lanes of the warp are converged (the four groups of a warp
// in lockstep).  A sub-warp mask held in a register makes nvcc guard every shuffle / vote with MATCH.ANY + REDUX + VOTEU + a divergence
// branch (~70 clk on the dependent chain, ~16 of them per level of the walk); with the literal 0xffffffff the guard disappears.
struct GrpW {
    static constexpr unsigned mask = 0xffffffffu;
    int lane; unsigned shift;
    __device__ __forceinline__ GrpW() {
        int l = threadIdx.x & 31;
        lane = l & 7;
        shift = (unsigned)(l & 24);
    }
    template <typename T> __device__ __forceinline__ T bcast(T v, int src) const { return __shfl_sync(0xffffffffu, v, src, 8); }
    __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(0xffffffffu, p) >> shift) & 0xffu; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};

__device__ __forceinline__ size_t node_at(const Arena &A, int g, int i) { return (size_t)g * A.M + i; }

// ------------------------------------------------------------------ exact arithmetic (see header comment)
__device__ __forceinline__ float ztab(const Arena &A, int n) {
    if (n >= 0 && n < ZTABLE_N) return A.ztable[n];
    double t = (double)n;                                   // special.h:26-33, evaluated in double
    double alpha = __dsub_rn(1.0, __ddiv_rn(1.0, t));
    double a = __ddiv_rn(-log(alpha), log(2.0));
    double b = __dsub_rn(1.0, __ddiv_rn(log(a), log(22.0)));
    return (float)__ddiv_rn(__dmul_rn(10.0, log(b)), log(41.0));   // core.h:93 narrows to float
}

// core.h:94 + core.h:213: q = (V[o] + score[c] - score[idx]) + z * sqrt(S2[o] / N[o]), all in float
__device__ __forceinline__ float clt_val(float V, float sc, float sidx) { return __fsub_rn(__fadd_rn(V, sc), sidx); }
__device__ __forceinline__ float clt_root(float S2, int N) { return __fsqrt_rn(__fdiv_rn(S2, (float)N)); }
__device__ __forceinline__ float clt_mix(float val, float z, float root) { return __fadd_rn(val, __fmul_rn(z, root)); }
__device__ __forceinline__ float clt_q(float V, float sc, float sidx, float z, float S2, int N) {
    return clt_mix(clt_val(V, sc, sidx), z, clt_root(S2, N));
}

// core.h:244-258, one trace level.  v is carried in double; stores narrow to float.
__device__ __forceinline__ void welford_level(int4 &st, double &v, double var, float score_idx, double gamma) {
    v = __dsub_rn(v, (double)score_idx);
    int n = st.x;
    float val = __int_as_float(st.y), s2 = __int_as_float(st.z);
    if (n == 0) {
        val = (float)v;
        s2 = (float)var;
    } else {
        double delta = __dsub_rn(v, (double)val);
        val = (float)__dadd_rn((double)val, __ddiv_rn(delta, (double)(n + 1)));
        double delta2 = __dsub_rn(v, (double)val);
        s2 = (float)__dadd_rn((double)s2, __ddiv_rn(__dsub_rn(__dmul_rn(delta, delta2), (double)s2), (double)(n + 1)));
    }
    st.x = n + 1; st.y = __float_as_int(val); st.z = __float_as_int(s2);
    v = __dadd_rn(__dmul_rn(gamma, v), (double)score_idx);
}

// ------------------------------------------------------------------ unique children (core.h:111-144)
// In: lane a (<7) holds child slot a as (c, o, s).  Out, per lane: is_first (this lane is the first occurrence of
// its observation: the list position), rep_c / rep_s = the child that represents the observation (the one with the
// strictly largest score, earliest on ties).
struct Uniq { bool is_first; int rep_c; float rep_s; unsigned first_mask; int rep_lane; };

template <typename G>
__device__ __forceinline__ Uniq unique_children(const G &gp, int c, int o, float s) {
    bool valid = gp.lane < 7 && c != 0;
    unsigned vmask = gp.ballot(valid);
    int first = -1, rep_c = 0, rep_lane = 0;
    float best = 0.f;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        int cj = gp.bcast(c, j), oj = gp.bcast(o, j);
        float sj = gp.bcast(s, j);
        if (((vmask >> j) & 1u) && oj == o) {
            if (first < 0) { first = j; best = sj; rep_c = cj; rep_lane = j; }
            else if (sj > best) { best = sj; rep_c = cj; rep_lane = j; }      // strict >, core.h:139
        }
    }
    Uniq u;
    u.is_first = valid && first == gp.lane;
    u.rep_c = rep_c; u.rep_s = best; u.rep_lane = rep_lane;
    u.first_mask = gp.ballot(u.is_first);
    return u;
}

// The child list of a node never changes once the node is expanded (children are linked once, the collector keeps every
// child of a reachable node), so core.h:111-144's de-duplication is done ONCE, when the expansion completes, and cached
// in the row: u[a] = representative child (28 bits) | lane of the representative << 28 | is_first << 31.
// select then needs no scan at all: one extra word from the same 128-byte line.
constexpr uint32_t LINK_NODE_MASK = 0x0fffffffu;
__device__ __forceinline__ uint32_t link_word(const Uniq &u) {
    return ((uint32_t)u.rep_c & LINK_NODE_MASK) | ((uint32_t)u.rep_lane << 28) | (u.is_first ? 0x80000000u : 0u);
}

// ------------------------------------------------------------------ cache-warming loads (see warm_expand)
// L2 residency hints (performance only).  One simulation step streams ~200 MB of activations (conv -> fc) and ~20 MB of new
// nodes through the 126 MB L2, so without hints nothing of the trees survives from one step to the next although every step
// re-walks the same top levels.  The first L2_HOT_LEVELS levels of every game's walk (row line + statistics, ~3.7 MB per
// level at 16384 games) are loaded / stored with an evict_last policy.
constexpr int L2_HOT_LEVELS = 16;
__device__ __forceinline__ uint64_t l2_policy(bool keep) {
    uint64_t last, normal;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(last));
    asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(normal));
    return keep ? last : normal;
}
__device__ __forceinline__ int32_t ldg_hint(const int32_t *p, uint64_t pol) {
    int32_t v;
    asm volatile("ld.global.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol) : "memory");
    return v;
}
__device__ __forceinline__ int4 ldg_hint(const int4 *p, uint64_t pol) {
    int4 v;
    asm volatile("ld.global.L2::cache_hint.v4.b32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol) : "memory");
    return v;
}
__device__ __forceinline__ void stg_hint(int4 *p, int4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
}

// non-blocking L2 prefetch: no destination register, so nothing ever waits for it (unlike the touch loads below)
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

__device__ __forceinline__ uint32_t touch32(const void *p) {
    uint32_t v;
    asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint2 touch64(const void *p) {
    uint2 v;
    asm volatile("ld.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}

// ------------------------------------------------------------------ path cache
// Consecutive simulations of a game walk almost the same path (CPU model in oracle/mcts_oracle.c: 90-94 % of the levels are a shared
// prefix; the walks differ in their last ~4 levels), and every level of a walk costs two DEPENDENT random accesses into an 82 GB arena.
// The walk therefore leaves, next to the trace, everything a level needs (sequential per game):
//   pc      [8 slots][trace_max] int4   slot a < 7: {link word u[a], val, visit, root} of child slot a AS OF THE WALK THAT FILLED THE LEVEL, where
//                                       val = (value + score) - own score and root = sqrt(variance / visit) are the two z-independent terms of
//                                       policy_clt's q = val + z * root (core.h:94, 213): stored as computed, so a cached sibling costs one
//                                       multiply-add pair instead of an IEEE division and square root (13 % of the kernel's samples in ncu);
//                                       slot 7: {0, own score, own observation, NODE id}
//   pc_var  [8 slots][trace_max] i32    slot a < 7: the score of the slot's representative child (to rebuild val of the picked slot from its live
//                                       statistics); slot 7: the slot the walk PICKED at this level (7: none)
//           (slot-major, level-minor: the cached levels are evaluated ONE LANE PER LEVEL, so the eight lanes of a game read eight consecutive
//            levels of one slot = one 128-byte line per load; level-major entries cost 32 wavefronts per load instruction and were slower)
//   pc_own  16 bytes per level          {visit, value, variance} of the level's own observation, rewritten by k_backup every simulation
//   pc_sib  16 bytes per level          the children's observation ids as 8 x u16 (0: not a first occurrence; the last: the picked slot),
//                                       read by k_backup's staleness scan only
// A level whose entry is valid and whose node id matches is served from the entry, with the picked child's statistics taken from the NEXT
// level's own record (the one statistic of the node's children that changes from simulation to simulation): same values, same
// arithmetic, same pick.  Coherence (the row fields of an expanded node never change; only statistics do, and only k_backup writes them
// for live observations):
//   * k_backup rewrites pc_own of every trace level (one coalesced 16-byte store per level);
//   * when a cached level picks another child than last time, the old pick's latest statistics go back into the entry first;
//   * any other copy — the same observation under another node of the path (transposition), or twice on the trace — goes stale:
//     k_backup finds those with a bitmap of the trace's own observations and truncates pc_len at the shallowest stale level;
//   * the entry of a leaf that gets expanded says "no children": the walk leaves pc_len = D - 1;
//   * k_update_root, k_gc (collections and dropped trees) and reset_tree set pc_len = 0.
// The CPU model applies exactly these rules and checks every value a cached level would read against the arena at every selection
// (oracle/mcts_oracle.c pc_*, tests/test_cpu_path_cache_model.py).
constexpr int PC_BYTES_PER_LEVEL = 8 * 16 + 8 * 4 + 16 + 16;   // pc + pc_var + pc_own + pc_sib
constexpr int PC_MAX_NODES = 65536;   // observation ids as u16 in pc_sib; k_backup's bitmap of the trace's observations is exact (one bit per slot, shared memory)
constexpr uint32_t TMETA_OBS_MASK = 0x0fffffffu;   // trace_meta.x = own observation | pick << 28

// ------------------------------------------------------------------ accessors
// The engine keeps the packed arena above; the single-call twins of agents/cppmodule/core.cpp:20-26 work on the
// reference's own array layout (agents/agent.py:58-88).  Both run the same select / backup code through these.
constexpr int ZS_N = 2048;   // z(n) entries staged in shared memory by k_select_expand (deep nodes have small n)

struct ArenaAcc {
    static constexpr bool has_pc = true;
    const Arena &A; int g; const float *zs;
    const int32_t *rowg; int4 *statg; int32_t *traceg; int2 *tmetag;   // this game's slices of the arena (address arithmetic hoisted out of the loops)
    int4 *pcg; int32_t *pvarg; uint16_t *psib; int4 *pown; int pc_len; // path cache of this game (nullptr: off) and its valid length for THIS walk (set by the caller)
    __device__ __forceinline__ ArenaAcc(const Arena &A_, int g_, const float *zs_ = nullptr)
        : A(A_), g(g_), zs(zs_), rowg(A_.row + (size_t)g_ * A_.M * ROW_WORDS), statg(A_.stat + (size_t)g_ * A_.M),
          traceg(A_.trace + (size_t)g_ * A_.trace_max), tmetag(A_.trace_meta + (size_t)g_ * A_.trace_max),
          pcg(A_.pc ? A_.pc + (size_t)g_ * A_.trace_max * 8 : nullptr), pvarg(A_.pc ? A_.pc_var + (size_t)g_ * A_.trace_max * 8 : nullptr),
          psib(A_.pc ? reinterpret_cast<uint16_t *>(A_.pc_sib + (size_t)g_ * A_.trace_max) : nullptr),
          pown(A_.pc ? A_.pc_own + (size_t)g_ * A_.trace_max : nullptr), pc_len(0) {}
    __device__ __forceinline__ int4 *pslot(int a, int L) const { return pcg + (size_t)a * A.trace_max + L; }
    __device__ __forceinline__ int32_t *pvar(int a, int L) const { return pvarg + (size_t)a * A.trace_max + L; }
    // the lines the NEXT round of eight levels (Lb .. Lb+7) will read, requested from L2 while this round is evaluated: lane a takes slot a
    __device__ __forceinline__ void pc_prefetch_round(int Lb, int lane) const {
        if (Lb >= A.trace_max) return;
        const int Le = Lb + 7 < A.trace_max ? Lb + 7 : A.trace_max - 1;
        prefetch_l2(pslot(lane, Lb)); prefetch_l2(pslot(lane, Le));
        prefetch_l2(pvar(lane, Lb));
        if (lane == 0) { prefetch_l2(pown + (Lb + 1 < A.trace_max ? Lb + 1 : Lb)); prefetch_l2(pown + Le); }
    }
    // One cached level, evaluated by ONE lane: check_low + policy_clt (core.h:65-105) over the seven child slots in list order, on the entry's
    // values with the slot picked last time read from the next level's own record.  Same float operations per child as clt_q in the
    // eight-lane form; the argmax is the reference's own loop (first entry, then strict >).  bail: a first child below `low` visits.
    __device__ __forceinline__ void pc_eval(int L, int low, int &node, int &own_obs, float &s_idx, int &pick_prev, int &pick, int &next,
                                            bool &leaf, bool &bail, int4 &wb) const {
        const int4 l7 = *pslot(7, L);
        pick_prev = *pvar(7, L);
        const int4 own = pown[L + 1 < A.trace_max ? L + 1 : L];
        s_idx = __int_as_float(l7.y); own_obs = l7.z; node = l7.w;
        const int pp = pick_prev < 7 ? pick_prev : 0;
        const float rep_s_p = __int_as_float(*pvar(pp, L));            // score of the picked slot's representative child (in flight with the slots below)
        int n = 0; unsigned fm = 0u; bool lowhit = false;
#pragma unroll
        for (int a = 0; a < 7; ++a) {                                   // pass 1: which slots are list entries, accumulate(visit) (core.h:88), check_low
            const int4 e = *pslot(a, L);
            const int vis = a == pick_prev ? own.x : e.z;
            if ((uint32_t)e.x >> 31) { fm |= 1u << a; n += vis; lowhit |= vis < low; }
        }
        leaf = fm == 0u; bail = lowhit;
        pick = 7; next = 0;
        if (leaf || lowhit) return;
        // the one child whose statistics moved since the entry was filled: its two z-independent terms from the live record, ONCE (inside the
        // unrolled loop below the division / square root were instantiated seven times: 1 280 instructions per round, 39 % of the kernel's)
        const float val_p = clt_val(__int_as_float(own.y), rep_s_p, s_idx);
        const float root_p = clt_root(__int_as_float(own.z), own.x);
        wb = make_int4(__float_as_int(val_p), own.x, __float_as_int(root_p), 0);
        const float zq = z(n);
        float bestq = 0.f;
#pragma unroll
        for (int a = 0; a < 7; ++a) {                                   // pass 2, branch free (the lines are in L1 now): q of every list entry, first strict maximum
            const int4 e = *pslot(a, L);
            const float val = a == pick_prev ? val_p : __int_as_float(e.y);
            const float root = a == pick_prev ? root_p : __int_as_float(e.w);
            const float q = clt_mix(val, zq, root);
            const bool take = ((fm >> a) & 1u) && (pick == 7 || q > bestq);   // core.h:94-101: first entry, then the first strict maximum
            pick = take ? a : pick;
            bestq = take ? q : bestq;
            next = take ? (int)((uint32_t)e.x & LINK_NODE_MASK) : next;
        }
    }
    // this lane's cached level picked another child than last time: the old pick's latest statistics return to the entry, the new pick is recorded
    __device__ __forceinline__ void pc_repick_lane(int L, int old_pick, int new_pick, const int4 &st) const {   // st = {val, visit, root} of the old pick as evaluated now
        uint8_t *e = reinterpret_cast<uint8_t *>(pslot(old_pick, L));
        *reinterpret_cast<int *>(e + 4) = st.x;
        *reinterpret_cast<int2 *>(e + 8) = make_int2(st.y, st.z);
        *pvar(7, L) = new_pick;
        psib[(size_t)L * 8 + 7] = (uint16_t)new_pick;
    }
    __device__ __forceinline__ void pc_store(int L, int lane, int4 e, int var, uint16_t sib) const {
        *pslot(lane, L) = e;
        *pvar(lane, L) = var;
        psib[(size_t)L * 8 + lane] = sib;
    }
    __device__ __forceinline__ void children(int idx, int lane, int &c, int &o, float &s) const {
        const int32_t *row = rowg + (size_t)idx * ROW_WORDS;
        c = row[lane]; o = row[8 + lane]; s = __int_as_float(row[16 + lane]);   // lane 7: own episode / obs / score
    }
    __device__ __forceinline__ void meta(int idx, int &o, float &s) const {
        const int32_t *row = rowg + (size_t)idx * ROW_WORDS;
        o = row[15]; s = __int_as_float(row[23]);
    }
    // one level of select: observation of this lane's child, the node's own score, the cached de-duplication.  `on` = this lane's group
    // is still walking (the loads are predicated, the shuffles are executed by every lane: see GrpW)
    template <typename G>
    __device__ __forceinline__ void level(const G &gp, bool on, int idx, int depth, int &o, float &s_idx, Uniq &u, float &s, uint32_t &lw) const {
        const int32_t *row = rowg + (size_t)idx * ROW_WORDS + gp.lane;
        s = 0.f; lw = 0u;
        o = 0;
        if (on) {
            const uint64_t pol = l2_policy(depth < L2_HOT_LEVELS);
            o = ldg_hint(row + 8, pol);
            s = __int_as_float(ldg_hint(row + 16, pol));
            lw = (uint32_t)ldg_hint(row + 24, pol);
        }
        s_idx = gp.bcast(s, 7);
        u.is_first = lw >> 31; u.rep_lane = (int)((lw >> 28) & 7u); u.rep_c = (int)(lw & LINK_NODE_MASK);
        u.rep_s = gp.bcast(s, u.rep_lane);
        u.first_mask = gp.ballot(u.is_first);
    }
    __device__ __forceinline__ int4 stat(int o) const { return statg[o]; }
    __device__ __forceinline__ void set_stat(int o, int4 st) const { statg[o] = st; }
    // the same, for a node at `depth` of the current walk (see L2_HOT_LEVELS)
    __device__ __forceinline__ int4 stat(int o, int depth) const { return ldg_hint(statg + o, l2_policy(depth < L2_HOT_LEVELS)); }
    __device__ __forceinline__ void set_stat(int o, int4 st, int depth) const { stg_hint(statg + o, st, l2_policy(depth < L2_HOT_LEVELS)); }
    __device__ __forceinline__ void meta(int idx, int depth, int &o, float &s) const {
        const int32_t *row = rowg + (size_t)idx * ROW_WORDS;
        const uint64_t pol = l2_policy(depth < L2_HOT_LEVELS);
        o = ldg_hint(row + 15, pol); s = __int_as_float(ldg_hint(row + 23, pol));
    }
    __device__ __forceinline__ void put_trace(int d, int idx) const { traceg[d] = idx; }
    __device__ __forceinline__ int get_trace(int d) const { return traceg[d]; }
    __device__ __forceinline__ void put_trace_meta(int d, int o, float s) const { tmetag[d] = make_int2(o, __float_as_int(s)); }
    __device__ __forceinline__ void get_trace_meta(int d, int &o, float &s) const { const int2 m = tmetag[d]; o = m.x & (int)TMETA_OBS_MASK; s = __int_as_float(m.y); }
    __device__ __forceinline__ void get_trace_meta_raw(int d, int &oraw, float &s) const { const int2 m = tmetag[d]; oraw = m.x; s = __int_as_float(m.y); }   // with the pick in bits 28-30
    __device__ __forceinline__ uint32_t rand() const { uint32_t sr = A.srng[g]; uint32_t r = rng_next(sr); A.srng[g] = sr; return r; }
    __device__ __forceinline__ float z(int n) const { return (zs && n >= 0 && n < ZS_N) ? zs[n] : ztab(A, n); }
};

struct RefAcc {   // child int32[M,7], visit int32[M], value/variance/score f32[M], n_to_o int32[M]  (core.cpp:20-26)
    static constexpr bool has_pc = false;
    static constexpr int4 *pcg = nullptr; static constexpr int pc_len = 0;
    __device__ __forceinline__ void pc_eval(int, int, int &, int &, float &, int &, int &, int &, bool &, bool &, int4 &) const {}
    __device__ __forceinline__ void pc_store(int, int, int4, int, uint16_t) const {}
    __device__ __forceinline__ void pc_repick_lane(int, int, int, const int4 &) const {}
    __device__ __forceinline__ void pc_prefetch_round(int, int) const {}
    const int32_t *child; int32_t *visit; float *value; float *variance; const float *score; const int32_t *n2o;
    int32_t *trace; uint32_t *rng; const Arena *A;
    __device__ __forceinline__ void children(int idx, int lane, int &c, int &o, float &s) const {
        if (lane < 7) { c = child[(size_t)idx * 7 + lane]; o = n2o[c]; s = score[c]; }
        else { c = 0; o = n2o[idx]; s = score[idx]; }
    }
    __device__ __forceinline__ void meta(int idx, int &o, float &s) const { o = n2o[idx]; s = score[idx]; }
    template <typename G>
    __device__ __forceinline__ void level(const G &gp, bool on, int idx, int, int &o, float &s_idx, Uniq &u, float &s, uint32_t &lw) const {
        int c = 0;
        s = 0.f; lw = 0u;
        o = 0;
        if (on) children(idx, gp.lane, c, o, s);
        s_idx = gp.bcast(s, 7);
        u = unique_children(gp, c, o, s);
    }
    __device__ __forceinline__ int4 stat(int o, int = 0) const { return make_int4(visit[o], __float_as_int(value[o]), __float_as_int(variance[o]), 0); }
    __device__ __forceinline__ void set_stat(int o, int4 st) const { visit[o] = st.x; value[o] = __int_as_float(st.y); variance[o] = __int_as_float(st.z); }
    __device__ __forceinline__ void put_trace(int d, int idx) const { trace[d] = idx; }
    __device__ __forceinline__ int get_trace(int d) const { return trace[d]; }
    __device__ __forceinline__ void put_trace_meta(int, int, float) const {}
    __device__ __forceinline__ uint32_t rand() const { uint32_t sr = *rng; uint32_t r = rng_next(sr); *rng = sr; return r; }
    __device__ __forceinline__ float z(int n) const { return ztab(*A, n); }
};

// ------------------------------------------------------------------ select (core.h:167-224)
// Returns the leaf; writes the trace.  All 8 lanes return the same values.
// Warp-lockstep walk: the four 8-lane groups of a warp descend their four trees level by level TOGETHER, all 32 lanes converged, so
// that every shuffle and vote carries the literal full mask (GrpW).  `active` = this lane's group has a tree to walk; a group that
// has reached its leaf idles (predicated) until the deepest of the four is done.  Returns the leaf; writes the trace; all 8 lanes of
// a group return the same values.  The whole warp must call this together.
template <typename Acc>
__device__ __forceinline__ int select_trace(const Acc &acc, bool active, int root, int low, int trace_max, int &D_out, int &status, int *cached_levels = nullptr) {
    const GrpW gp;
    int idx = root, D = 0;
    bool walking = active;
    // core.h:65-105 for one level, from the values every lane holds for its child slot (`on`: this lane's group is at a node WITH children):
    // check_low, then policy_clt.  Shared by the cached and the uncached form of a level, so both pick bit for bit the same child.
    auto choose = [&](bool on, const Uniq &u, const int4 &st, float s_idx, float &val_out, float &root_out) -> int {
        const unsigned lowmask = gp.ballot(on && u.is_first && st.x < low);   // core.h:65-77
        int pick = 0;
        if (__any_sync(0xffffffffu, lowmask != 0u)) {                   // warp-uniform branch: the draw of every group that needs one
            uint32_t r = 0;
            if (lowmask != 0u && gp.lane == 0) r = acc.rand();
            r = gp.bcast(r, 0);
            if (lowmask != 0u) pick = (int)__fns(lowmask, 0, (int)(r % (uint32_t)__popc(lowmask)) + 1);
        }
        int n = (on && u.is_first) ? st.x : 0;                          // core.h:88 accumulate(visit)
        n += __shfl_xor_sync(0xffffffffu, n, 1, 8);
        n += __shfl_xor_sync(0xffffffffu, n, 2, 8);
        n += __shfl_xor_sync(0xffffffffu, n, 4, 8);
        const float z = acc.z(n);
        const bool cmp = on && u.is_first;
        val_out = cmp ? clt_val(__int_as_float(st.y), u.rep_s, s_idx) : 0.f;
        root_out = cmp ? clt_root(__int_as_float(st.z), st.x) : 0.f;
        const float q = cmp ? clt_mix(val_out, z, root_out) : 0.f;
        // core.h:94-101: the first strict maximum in list order = the largest q, the lowest lane on ties, as a 3-step
        // butterfly.  A NaN never wins a `>`; it is the answer only when it is the first entry of the list.
        const bool cand = cmp && q == q;
        float qv = cand ? q : -INFINITY;
        int ql = cand ? gp.lane : 8 + gp.lane;                           // non-candidates lose every tie
#pragma unroll
        for (int d = 1; d < 8; d <<= 1) {
            const float oq = __shfl_xor_sync(0xffffffffu, qv, d, 8);
            const int ol = __shfl_xor_sync(0xffffffffu, ql, d, 8);
            const bool take = oq > qv || (oq == qv && ol < ql);
            qv = take ? oq : qv; ql = take ? ol : ql;
        }
        const int first = __ffs(u.first_mask) - 1;
        const unsigned nanmask = gp.ballot(cmp && q != q);
        if (lowmask == 0u) pick = (first >= 0 && ((nanmask >> first) & 1u)) ? first : ql;
        return pick;
    };
    if constexpr (Acc::has_pc) {
        // ---- phase 1: the levels the path cache still holds (see "path cache" above), ONE LANE PER LEVEL.  Given its entry and the next
        // level's own record, the pick of a cached level does not depend on the levels above it, so the eight lanes of a group evaluate
        // eight consecutive levels at once, each lane running core.h:83-105 over the seven child slots serially (no shuffles: ~9 x fewer
        // warp instructions per level than eight lanes per level, which was issue bound at ~1.5 k clk per level).  The walk follows the
        // cached path up to the first level that picks another child than last time (served, with the new pick), is a leaf (served: the
        // walk ends), or cannot be served (entry missing, a child below `low` visits: check_low draws from the RNG in the uncached form).
        const int pcl = (walking && acc.pcg) ? acc.pc_len : 0;          // group-uniform
        bool fast = pcl > 0;
        int n_cached = 0;
        while (__any_sync(0xffffffffu, fast)) {
            const int L = D + gp.lane;                                  // this lane's level
            const bool have = fast && L < pcl;
            int e_node = 0, e_own = 0, pick_prev = 7, pick = 7, next = 0; float s_idx = 0.f;
            bool leaf = false, bail = false;
            int4 wb = make_int4(0, 0, 0, 0);                            // the old pick's statistics as read here (written back if the pick changes)
            if (fast && D + 8 < pcl) acc.pc_prefetch_round(D + 8, gp.lane);
            if (have) acc.pc_eval(L, low, e_node, e_own, s_idx, pick_prev, pick, next, leaf, bail, wb);
            // the chain: level D must be the node the walk stands on, level L > D the child level L - 1 picks (true by construction while no pick changes)
            const int prev_next = __shfl_up_sync(0xffffffffu, next, 1, 8);
            const int expect = gp.lane == 0 ? idx : prev_next;
            if (have && e_node != expect) bail = true;
            const bool changed = have && !leaf && !bail && pick != pick_prev;
            // (every shuffle / vote below is executed by all 32 lanes, unconditionally: the four groups of a warp are in different states, and a
            // full-mask collective that only some groups reach never completes — session 26/27 hung on a `first < 8 && ballot(...)`)
            const unsigned stopmask = gp.ballot(!have || bail || leaf || changed);
            const unsigned okmask = gp.ballot(have && !bail);
            const int first = stopmask ? __ffs(stopmask) - 1 : 8;       // lanes below `first`: served, pick unchanged
            const bool first_served = first < 8 && ((okmask >> first) & 1u) != 0u;   // the stopping level itself: a leaf or a changed pick
            const int served = first + (first_served ? 1 : 0);
            const int last_next = gp.bcast(next, served > 0 ? served - 1 : 0);
            const int leaf_at_first = gp.bcast(leaf ? 1 : 0, first < 8 ? first : 0);
            const int leaf_node = gp.bcast(e_node, first < 8 ? first : 0);
            const bool ended = first_served && leaf_at_first != 0;
            if (fast) {
                if (gp.lane < served) {
                    acc.put_trace_meta(L, e_own | (leaf ? 0 : pick << 28), s_idx);
                    if (changed) acc.pc_repick_lane(L, pick_prev, pick, wb);
                }
                n_cached += served;
                D += served;
                if (ended) idx = leaf_node;                             // the walk returns the leaf it stands on
                else if (served > 0) idx = last_next;
                if (ended) { walking = false; fast = false; }           // core.h:200: a cached leaf without children (terminal node)
                else if (first < 8 || D >= pcl) fast = false;           // uncached from level D on
            }
        }
        if (cached_levels) *cached_levels = n_cached;
    }
    // ---- phase 2: uncached levels (two dependent random accesses each); with the path cache on, each of them leaves its entry behind
    while (__any_sync(0xffffffffu, walking)) {
        if (walking && D >= trace_max) { status = ST_TRACE_FULL; walking = false; }
        if (walking) {
            if (gp.lane == 0) acc.put_trace(D, idx);
            ++D;
        }
        const bool at_level = walking;                                  // this group loads level D - 1 in this round
        int o; float s_idx, s_own; uint32_t lw;
        Uniq u;
        acc.level(gp, walking, idx, D - 1, o, s_idx, u, s_own, lw);
        if (u.first_mask == 0) walking = false;                         // core.h:200 no children: leaf (group-uniform)
        int4 st = make_int4(0, 0, 0, 0);
        if (walking && u.is_first) st = acc.stat(o, D);                 // the children live one level below
        float q_val, q_root;
        const int pick = choose(walking, u, st, s_idx, q_val, q_root);
        const int next = gp.bcast(u.rep_c, pick);
        if (at_level && gp.lane == 7) acc.put_trace_meta(D - 1, o | (walking ? pick << 28 : 0), s_idx);   // lane 7 holds the node's own observation and score
        if constexpr (Acc::has_pc) {
            if (at_level && acc.pcg) {
                const int pk = walking ? pick : 7;
                acc.pc_store(D - 1, gp.lane, gp.lane == 7 ? make_int4(0, __float_as_int(s_own), o, idx) : make_int4((int)lw, __float_as_int(q_val), st.x, __float_as_int(q_root)),
                             gp.lane == 7 ? pk : __float_as_int(u.rep_s), gp.lane == 7 ? (uint16_t)pk : (uint16_t)(u.is_first ? o : 0));
            }
        }
        if (walking) idx = next;
    }
    __syncwarp();
    D_out = D;
    return idx;
}

// ------------------------------------------------------------------ hash tables
__device__ __forceinline__ uint32_t fold32(uint64_t h) { uint32_t x = (uint32_t)(h ^ (h >> 32)); return x ? x : 1u; }
// open addressing over H slots, H any size (1.5 x max_nodes: a power of two would cost up to 2.67 x): home slot by multiply-shift, linear probing
__device__ __forceinline__ uint32_t tab_home(uint32_t h, int H) { return __umulhi(h, (uint32_t)H); }
__device__ __forceinline__ uint32_t tab_next(uint32_t p, int H) { return p + 1u == (uint32_t)H ? 0u : p + 1u; }

// Find `words` (nw of them, held identically by every lane) in a table whose entries index `store` records.
// Group-cooperative: lane j compares uint4 j of the candidate record.  Returns index or 0.
template <int NW>
__device__ __forceinline__ int table_find(const Grp &gp, const uint2 *tab, int H, const uint32_t *store, size_t base,
                                          const uint32_t (&words)[NW], uint32_t h, int *slot_out = nullptr) {
    uint32_t p = tab_home(h, H);
    for (;;) {
        uint2 e = tab[p];
        if (e.y == 0u) return 0;
        if (e.y != 0xffffffffu && e.x == h) {
            bool eq = true;
            if (gp.lane * 4 < NW) {
                const uint4 v = *reinterpret_cast<const uint4 *>(store + (base + e.y) * NW + gp.lane * 4);
                int k = gp.lane * 4;
                // words[] is indexed with a lane-dependent offset; unrolled selects keep it in registers
                uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
                for (int q = 0; q < NW / 4; ++q)
                    if (q * 4 == k) { a0 = words[q * 4]; a1 = words[q * 4 + 1]; a2 = words[q * 4 + 2]; a3 = words[q * 4 + 3]; }
                eq = v.x == a0 && v.y == a1 && v.z == a2 && v.w == a3;
            }
            if (gp.ballot(eq) == 0xffu) { if (slot_out) *slot_out = (int)p; return (int)e.y; }
        }
        p = tab_next(p, H);
    }
}

__device__ __forceinline__ void table_insert(const Grp &gp, uint2 *tab, int H, uint32_t h, int idx) {
    if (gp.lane == 0) {
        uint32_t p = tab_home(h, H);
        for (;;) {
            uint32_t y = tab[p].y;
            if (y == 0u || y == 0xffffffffu) break;
            p = tab_next(p, H);
        }
        tab[p] = make_uint2(h, (uint32_t)idx);
    }
    gp.sync();
}

// ------------------------------------------------------------------ garbage collection (agent.py:187-257)
// remove_nodes runs as its own CTA-per-game kernel (kernels.cuh: k_gc): a game whose free list runs dry suspends
// its expansion at exactly the child where the reference would call remove_nodes (agent.py:96-97), the collection
// runs with a whole thread block, and k_expand_resume continues with the remaining children.

// ------------------------------------------------------------------ new_node (agent.py:90-130)
// `w` = packed game, held identically by all lanes.  Returns node index (0 on arena overflow); o_out/score_out are
// the node's observation and score (what the parent's row caches for it).
// Pre-digested game: what new_node needs besides the record itself.  expand_leaf computes it once per child, in parallel
// (lane a digests child a), instead of all eight lanes re-deriving every child's hashes and observation key in turn.
struct Digest { uint32_t h, hk; uint32_t key[KEY_WORDS]; int end; float score; };

__device__ __forceinline__ void digest_game(const uint32_t (&w)[REC_WORDS], Digest &d) {
    d.h = fold32(hash_words(w, REC_WORDS));
    Game gm;
    unpack(gm, w);
    obskey(gm, d.key);
    d.hk = fold32(hash_words(d.key, KEY_WORDS));
    d.end = gm.end;
    d.score = (float)gm.score;                                              // agent.py:106 score[idx] = game.score
}

// n_new: where to count a created node (group-uniform register, flushed by the caller); nullptr = count in A.counters[6] here.
__device__ __forceinline__ int new_node(const Arena &A, const Grp &gp, int g, const uint32_t (&w)[REC_WORDS], const Digest &dg, int &o_out,
                                        float &score_out, int &status, bool may_suspend, int *n_new = nullptr) {
    const int M = A.M, H = A.H;
    uint2 *ntab = A.ntab + (size_t)g * H;
    const uint32_t h = dg.h;
    int idx = table_find<REC_WORDS>(gp, ntab, H, A.rec, (size_t)g * M, w, h);
    int32_t *rowb = A.row + (size_t)g * M * ROW_WORDS;
    if (idx) {
        o_out = rowb[(size_t)idx * ROW_WORDS + 15];
        score_out = __int_as_float(rowb[(size_t)idx * ROW_WORDS + 23]);
        return idx;
    }
    int nf = A.n_nfree[g];
    if (nf == 0) {      // agent.py:96-97: remove_nodes() is due here.  First time: suspend for k_gc; after it: the arena is full.
        status = may_suspend ? ST_NEED_GC : ST_ARENA_FULL; o_out = 0; score_out = 0.f; return 0;
    }
    idx = A.nfree[(size_t)g * M + nf - 1];                                  // agent.py:99 pop() from the right
    gp.sync();
    if (gp.lane == 0) A.n_nfree[g] = nf - 1;
    if (gp.lane < 5) {
        uint4 v;
        int k = gp.lane * 4;
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
        for (int q = 0; q < 5; ++q) if (q * 4 == k) { a0 = w[q * 4]; a1 = w[q * 4 + 1]; a2 = w[q * 4 + 2]; a3 = w[q * 4 + 3]; }
        v = make_uint4(a0, a1, a2, a3);
        *reinterpret_cast<uint4 *>(A.rec + ((size_t)g * M + idx) * REC_WORDS + k) = v;
    }
    gp.sync();
    table_insert(gp, ntab, H, h, idx);
    // observation (agent.py:114-128)
    const uint32_t (&key)[KEY_WORDS] = dg.key;
    const uint32_t hk = dg.hk;
    uint2 *otab = A.otab + (size_t)g * H;
    int o = table_find<KEY_WORDS>(gp, otab, H, A.key, (size_t)g * M, key, hk);
    if (!o) {
        int nof = A.n_ofree[g];
        o = A.ofree[(size_t)g * M + nof - 1];
        gp.sync();
        if (gp.lane == 0) {
            A.n_ofree[g] = nof - 1;
            A.stat[node_at(A, g, o)] = make_int4(0, 0, 0, dg.end);
        }
        if (gp.lane >= 1 && gp.lane < 4) {
            int k = (gp.lane - 1) * 4;
            uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
            for (int q = 0; q < 3; ++q) if (q * 4 == k) { a0 = key[q * 4]; a1 = key[q * 4 + 1]; a2 = key[q * 4 + 2]; a3 = key[q * 4 + 3]; }
            *reinterpret_cast<uint4 *>(A.key + ((size_t)g * M + o) * KEY_WORDS + k) = make_uint4(a0, a1, a2, a3);
        }
        gp.sync();
        table_insert(gp, otab, H, hk, o);
    }
    const float sc = dg.score;
    if (gp.lane == 7) {
        int32_t *r = rowb + (size_t)idx * ROW_WORDS;
        r[7] = A.episode[g]; r[15] = o; r[23] = __float_as_int(sc);
    }
    if (n_new) *n_new += 1;
    if (gp.lane == 0) {
        if (!n_new) atomicAdd(&A.counters[6], 1ull);
        if (A.nstat) A.nstat[node_at(A, g, idx) * NSTAT_WORDS + 2] = sc;   // node_stats[idx][2] = reward (core_distributional.py:86,112)
    }
    gp.sync();
    o_out = o; score_out = sc;
    return idx;
}

__device__ __forceinline__ int new_node(const Arena &A, const Grp &gp, int g, const uint32_t (&w)[REC_WORDS], int &o_out,
                                        float &score_out, int &status, bool may_suspend) {
    Digest dg;
    digest_game(w, dg);
    return new_node(A, gp, g, w, dg, o_out, score_out, status, may_suspend);
}

// ------------------------------------------------------------------ overflow policy (beyond the reference)
// When the reachable set alone fills the arena the reference dies (IndexError at agent.py:99 / UB at agent.cpp:227-231).
// With overflow_reset the tree of that game is dropped and re-rooted at the live game: statistics restart as at the
// first move of an episode.  Never taken when the arena is sized like the reference's (tests run with it off).
__device__ __noinline__ void reset_tree(const Arena &A, const Grp &gp, int g, int &status) {
    const int M = A.M, H = A.H;
    if (A.pc && gp.lane == 0) A.pc_len[g] = 0;     // path cache: the tree is gone
    if (status != ST_RESET_DONE) {        // (k_gc has already cleared the arena with a whole thread block in that case)
        int4 *rows = reinterpret_cast<int4 *>(A.row + (size_t)g * M * ROW_WORDS);
        for (int i = gp.lane; i < M * (ROW_WORDS / 4); i += 8) rows[i] = make_int4(0, 0, 0, 0);
        int4 *statb = A.stat + (size_t)g * M;
        for (int i = gp.lane; i < M; i += 8) statb[i] = make_int4(0, 0, 0, 0);
        uint4 *keyb = reinterpret_cast<uint4 *>(A.key + (size_t)g * M * KEY_WORDS);
        for (int i = gp.lane; i < M * 3; i += 8) keyb[i] = make_uint4(0, 0, 0, 0);
        uint2 *ntab = A.ntab + (size_t)g * H, *otab = A.otab + (size_t)g * H;
        for (int i = gp.lane; i < H; i += 8) { ntab[i] = make_uint2(0, 0); otab[i] = make_uint2(0, 0); }
        if (A.nstat) {
            float *ns = A.nstat + (size_t)g * M * NSTAT_WORDS, *nd = A.ndist + (size_t)g * M * A.dist_bins;
            for (int i = gp.lane; i < M * NSTAT_WORDS; i += 8) ns[i] = 0.f;
            for (size_t i = gp.lane; i < (size_t)M * A.dist_bins; i += 8) nd[i] = 0.f;
        }
        int32_t *nfree = A.nfree + (size_t)g * M, *ofree = A.ofree + (size_t)g * M;
        for (int i = gp.lane; i < M - 1; i += 8) { nfree[i] = i + 1; ofree[i] = i + 1; }
        if (gp.lane == 0) { A.n_nfree[g] = M - 1; A.n_ofree[g] = M - 1; atomicAdd(&A.counters[7], 1ull); }
    }
    gp.sync();
    status = ST_OK;
    uint32_t w[REC_WORDS];
#pragma unroll
    for (int q = 0; q < REC_WORDS / 4; ++q) {
        uint4 v = *reinterpret_cast<const uint4 *>(A.cur + (size_t)g * REC_WORDS + q * 4);
        w[q * 4] = v.x; w[q * 4 + 1] = v.y; w[q * 4 + 2] = v.z; w[q * 4 + 3] = v.w;
    }
    int o; float sc;
    int idx = new_node(A, gp, g, w, o, sc, status, false);
    if (gp.lane == 0) { A.root[g] = idx; A.status[g] = status; }
    gp.sync();
}

// ------------------------------------------------------------------ expand (agent.py:136-145)
// lane a plays action a on the leaf's game; the seven results are then inserted in action order (first seen wins,
// free-list order and a mid-expand garbage collection all as in the reference).  Leaves c/o/s of child a in lane a.
// Shared-memory staging of the seven children of one expansion: lane a plays action a, digests the resulting game and parks
// record | observation key | hashes in its slot; the insertion loop then reads child a with broadcast loads.  (Holding the
// 36 words per lane in registers across the loop and moving them with 36 shuffles per child spilled at 64 registers.)
// Cache warming (performance hint only; results discarded, so exactness is untouched).  One expansion is seven new_node calls in
// the reference's order, each a chain of dependent probes (node table -> record compare -> free list -> observation table ->
// key compare ...); at 16384 games the arenas span ~80 GB, every first touch is a DRAM access (~2.4 k clk measured) and the chain
// was ~50 of them per expansion.  Before the ordered loop, lane a touches everything child a's new_node will read first: its two
// table slots, then (on a hash match) the candidate record / row / key; lane 7 touches the counters and the free-list tails.  The
// ordered loop then runs on L1/L2 hits.  Real loads (volatile asm) are used: a prefetch instruction may be dropped.
__device__ __forceinline__ void warm_expand(const Arena &A, const Grp &gp, int g, uint32_t h, uint32_t hk) {
    const int M = A.M, H = A.H;
    if (gp.lane < 7) {
        const uint2 e1 = touch64(A.ntab + (size_t)g * H + tab_home(h, H));
        const uint2 e2 = touch64(A.otab + (size_t)g * H + tab_home(hk, H));
        if (e1.y != 0u && e1.y != 0xffffffffu && e1.x == h) {       // probable transposition: its record (80 B) and its row's own fields
            const uint32_t *r = A.rec + ((size_t)g * M + e1.y) * REC_WORDS;
            touch32(r); touch32(r + REC_WORDS - 1);
            touch32(A.row + ((size_t)g * M + e1.y) * ROW_WORDS + 15);
        }
        if (e2.y != 0u && e2.y != 0xffffffffu && e2.x == hk) {      // probable known observation: its key (48 B)
            const uint32_t *k = A.key + ((size_t)g * M + e2.y) * KEY_WORDS;
            touch32(k); touch32(k + KEY_WORDS - 1);
        }
    } else {
        const int nf = (int)touch32(A.n_nfree + g), nof = (int)touch32(A.n_ofree + g);
        touch32(A.episode + g);
        if (nf > 0) { touch32(A.nfree + (size_t)g * M + nf - 1); if (nf > 7) touch32(A.nfree + (size_t)g * M + nf - 7); }
        if (nof > 0) { touch32(A.ofree + (size_t)g * M + nof - 1); if (nof > 7) touch32(A.ofree + (size_t)g * M + nof - 7); }
    }
}

constexpr int STAGE_WORDS = 36;                      // rec[20] | key[12] | h, hk, end, score
constexpr int STAGE_GROUP_WORDS = 7 * STAGE_WORDS;   // per game in flight

__device__ __forceinline__ void expand_leaf(const Arena &A, const Grp &gp, int g, int leaf, const uint32_t (&leafrec)[REC_WORDS],
                                            int &c, int &o, float &s, int &status, int a_begin, bool may_suspend, int &a_stop,
                                            uint32_t *stage, int *n_new) {
    uint32_t wh = 0, whk = 0;
    if (gp.lane < 7) {
        uint32_t mine[REC_WORDS];
        Digest dm;
        Game gm;
        unpack(gm, leafrec);
        play(gm, gp.lane);
        pack(gm, mine);
        digest_game(mine, dm);
        uint4 *dst = reinterpret_cast<uint4 *>(stage + gp.lane * STAGE_WORDS);
#pragma unroll
        for (int q = 0; q < REC_WORDS / 4; ++q) dst[q] = make_uint4(mine[4 * q], mine[4 * q + 1], mine[4 * q + 2], mine[4 * q + 3]);
#pragma unroll
        for (int q = 0; q < KEY_WORDS / 4; ++q) dst[5 + q] = make_uint4(dm.key[4 * q], dm.key[4 * q + 1], dm.key[4 * q + 2], dm.key[4 * q + 3]);
        dst[8] = make_uint4(dm.h, dm.hk, (uint32_t)dm.end, __float_as_uint(dm.score));
        wh = dm.h; whk = dm.hk;
    }
    warm_expand(A, gp, g, wh, whk);
    gp.sync();
    c = 0; o = 0; s = 0.f;
    a_stop = N_ACTIONS;
    for (int a = a_begin; a < N_ACTIONS; ++a) {
        const uint4 *src = reinterpret_cast<const uint4 *>(stage + a * STAGE_WORDS);
        uint32_t w[REC_WORDS];
        Digest dg;
#pragma unroll
        for (int q = 0; q < REC_WORDS / 4; ++q) { const uint4 v = src[q]; w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w; }
#pragma unroll
        for (int q = 0; q < KEY_WORDS / 4; ++q) { const uint4 v = src[5 + q]; dg.key[4 * q] = v.x; dg.key[4 * q + 1] = v.y; dg.key[4 * q + 2] = v.z; dg.key[4 * q + 3] = v.w; }
        { const uint4 v = src[8]; dg.h = v.x; dg.hk = v.y; dg.end = (int)v.z; dg.score = __uint_as_float(v.w); }
        int oo; float ss;
        int idx = new_node(A, gp, g, w, dg, oo, ss, status, may_suspend, n_new);
        if (status == ST_NEED_GC) { a_stop = a; break; }     // resume at this child after k_gc
        if (gp.lane == a) { c = idx; o = oo; s = ss; }
        // agent.py:145 writes child[i] as soon as new_node returns, so a collection triggered by a later
        // sibling already sees this child as reachable
        if (gp.lane == a) {
            int32_t *r = A.row + node_at(A, g, leaf) * ROW_WORDS;
            r[a] = idx; r[8 + a] = oo; r[16 + a] = __float_as_int(ss);
        }
        gp.sync();
        if (status != ST_OK) break;
    }
    if (!n_new && gp.lane == 0 && status == ST_OK) atomicAdd(&A.counters[1], 1ull);   // with n_new the caller counts the expansion too
}

// ------------------------------------------------------------------ backup (core.h:226-260), one thread
template <typename Acc>
__device__ __forceinline__ void backup_trace(const Acc &acc, int D, double v, double var, double gamma) {
    for (int i = D - 1; i >= 0; --i) {
        int idx = acc.get_trace(i);
        int o; float sc;
        acc.meta(idx, o, sc);
        int4 st = acc.stat(o);
        welford_level(st, v, var, sc, gamma);
        acc.set_stat(o, st);
    }
}

// core.h:262-301 (the "mixture" update; not on the live path — ValueSimLP.py:29 passes mixture=False — kept for the
// single-call twin of backup_trace_obs_LP)
template <typename Acc>
__device__ __forceinline__ void backup_trace_mixture(const Acc &acc, int D, double v, double var, double gamma) {
    for (int i = D - 1; i >= 0; --i) {
        int idx = acc.get_trace(i);
        int o; float sc;
        acc.meta(idx, o, sc);
        int4 st = acc.stat(o);
        v = __dsub_rn(v, (double)sc);
        int n = st.x + 1;
        float val = __int_as_float(st.y), s2 = __int_as_float(st.z);
        double v_sq_diff = __dsub_rn(__dmul_rn(v, v), (double)__fmul_rn(val, val));
        double v_tmp = (double)val;
        double delta = __ddiv_rn(__dsub_rn(v, (double)val), (double)n);
        val = (float)__dadd_rn((double)val, delta);
        double var_diff = __dsub_rn(var, (double)s2);
        double upd = __dsub_rn(__ddiv_rn(__dadd_rn(var_diff, v_sq_diff), (double)n), __dmul_rn(delta, __dadd_rn(v_tmp, (double)val)));
        s2 = (float)__dadd_rn((double)s2, upd);
        st.x = n; st.y = __float_as_int(val); st.z = __float_as_int(s2);
        acc.set_stat(o, st);
        v = __dadd_rn(__dmul_rn(gamma, v), (double)sc);
        var = __dmul_rn(var, __dmul_rn(gamma, gamma));
    }
}

// core.h:303-381 leaf-parallel initialise + (averaged | per-child) backup, one thread.
//   c_nodes/c_obs: the unique children of the leaf (core.h:111-144 order); ev/evar: evaluator outputs per child;
//   child_end[i]: the `end` flag the reference tests for child i (SURVEY N1: the Python path passes the never-written
//   node array => all false; agent.cpp:538 tests the observation's flag).
template <typename Acc>
__device__ __forceinline__ void lp_backup(const Acc &acc, int D, int k, const int *c_obs, const float *c_score,
                                          const float *ev, const float *evar, const bool *child_end, double gamma,
                                          bool mixture, bool averaged, bool var_gamma2, float leaf_score) {
    if (k > 0) {
        double v_tmp = 0.0, var_tmp = 0.0;
        for (int i = 0; i < k; ++i) {
            int4 st = acc.stat(c_obs[i]);
            if (st.x == 0) {                                               // core.h:344-353
                st.x = 1;
                if (child_end[i]) { st.y = __float_as_int(0.f); st.z = __float_as_int(0.f); }
                else { st.y = __float_as_int(ev[i]); st.z = __float_as_int(evar[i]); }
                acc.set_stat(c_obs[i], st);
            }
            float val = __int_as_float(st.y), s2 = __int_as_float(st.z);
            if (averaged) {                                                // core.h:354-356
                v_tmp = __dadd_rn(v_tmp, __dadd_rn((double)c_score[i], __dmul_rn(gamma, (double)val)));
                var_tmp = __dadd_rn(var_tmp, (double)s2);
            } else {                                                       // core.h:357-361 (value + gamma*score, as written)
                double bv = __dadd_rn((double)val, __dmul_rn(gamma, (double)c_score[i]));
                double bvar = __dmul_rn(__dmul_rn(gamma, gamma), (double)s2);
                if (mixture) backup_trace_mixture(acc, D, bv, bvar, gamma);
                else backup_trace(acc, D, bv, bvar, gamma);
            }
        }
        if (averaged) {
            v_tmp = __ddiv_rn(v_tmp, (double)k);                           // core.h:364
            if (var_gamma2) var_tmp = __dmul_rn(var_tmp, __ddiv_rn(__dmul_rn(gamma, gamma), (double)k));   // core.h:365
            else {                                                         // agent.cpp:557-562: /k, then float arguments
                var_tmp = __ddiv_rn(var_tmp, (double)k);
                v_tmp = (double)(float)v_tmp; var_tmp = (double)(float)var_tmp;
            }
            if (mixture) backup_trace_mixture(acc, D, v_tmp, var_tmp, gamma);
            else backup_trace(acc, D, v_tmp, var_tmp, gamma);
        }
    } else {                                                               // core.h:368-371 terminal leaf
        if (mixture) backup_trace_mixture(acc, D, (double)leaf_score, 0.0, gamma);
        else backup_trace(acc, D, (double)leaf_score, 0.0, gamma);
    }
}

// ------------------------------------------------------------------ distributional select (core_distributional.py:82-106)
// Group form of dist_dev.cuh: dist_select_trace on the packed arena.  Unique children are ordered by ascending node index
// (the documented stand-in for numba's set order); lane a holds child slot a.
__device__ __forceinline__ double dist_z(double n) {
    double alpha = 1.0 - 1.0 / n;
    return 10.0 * log(1.0 - log(-log(alpha) / log(2.0)) / log(22.0)) / log(41.0);
}

__device__ __forceinline__ int dist_select_group(const Arena &A, const Grp &gp, int g, int root, int &D_out, int &status) {
    int idx = root, D = 0;
    const float *nsb = A.nstat + (size_t)g * A.M * NSTAT_WORDS;
    for (;;) {
        if (D >= A.trace_max) { status = ST_TRACE_FULL; break; }
        if (gp.lane == 0) A.trace[(size_t)g * A.trace_max + D] = idx;
        ++D;
        const int32_t *row = A.row + node_at(A, g, idx) * ROW_WORDS;
        int c = gp.lane < 7 ? row[gp.lane] : 0;
        bool uniq = c != 0;
        int rank = 0;                                    // position of this child in ascending-index order among the unique ones
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            int cj = gp.bcast(c, j);
            if (cj != 0 && cj == c && j < gp.lane) uniq = false;
        }
        unsigned umask = gp.ballot(uniq);
        if (umask == 0) break;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            int cj = gp.bcast(c, j);
            if (((umask >> j) & 1u) && cj < c) ++rank;
        }
        float4 ns = make_float4(0.f, 0.f, 0.f, 0.f);
        if (uniq) ns = *reinterpret_cast<const float4 *>(nsb + (size_t)c * NSTAT_WORDS);    // visit, mean, reward, variance
        const double r = (double)nsb[(size_t)idx * NSTAT_WORDS + 2];
        unsigned lowmask = gp.ballot(uniq && ns.x < (float)A.low);
        int pick_lane = -1;
        if (lowmask) {                                   // agents/core.py:462-468 check_low: uniform pick among the low children
            uint32_t x = 0;
            if (gp.lane == 0) { uint32_t sr = A.srng[g]; x = rng_next(sr); A.srng[g] = sr; }
            x = gp.bcast(x, 0);
            int want = (int)(x % (uint32_t)__popc(lowmask));
            int lrank = 0;
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                int cj = gp.bcast(c, j);
                if (((lowmask >> j) & 1u) && cj < c) ++lrank;
            }
            pick_lane = __ffs(gp.ballot(((lowmask >> gp.lane) & 1u) && lrank == want)) - 1;
        } else {                                         // policy_dist, core_distributional.py:66-79
            double n = uniq ? (double)ns.x : 0.0;        // visits are integers: the double sum is exact in any order
            n += __shfl_xor_sync(gp.mask, n, 1, 8); n += __shfl_xor_sync(gp.mask, n, 2, 8); n += __shfl_xor_sync(gp.mask, n, 4, 8);
            const double z = dist_z(n);
            float s0 = (float)((double)__fadd_rn(ns.y, ns.z) - r);
            float s1 = (float)((double)ns.w / ((double)ns.x + 1e-3));
            double q = (double)s0 + z * (double)__fsqrt_rn(s1);
            double bq = 0.0;
            const int k = __popc(umask);
            for (int rr = 0; rr < k; ++rr) {             // np.argmax over the ascending list: first maximum
                int L = __ffs(gp.ballot(uniq && rank == rr)) - 1;
                double qL = gp.bcast(q, L);
                if (rr == 0 || qL > bq) { bq = qL; pick_lane = L; }
            }
        }
        idx = gp.bcast(c, pick_lane);
    }
    D_out = D;
    return idx;
}

// Scalar form of core.h:111-144 for one thread (backup side): fills c_obs / c_score(rep) / first-slot list.
template <typename Acc>
__device__ __forceinline__ int unique_scalar(const Acc &acc, int idx, int *c_nodes, int *c_obs, float *c_score, int *slot) {
    int k = 0;
    for (int a = 0; a < 7; ++a) {
        int c, o; float s;
        acc.children(idx, a, c, o, s);
        if (c == 0) continue;
        int j = 0;
        while (j < k && c_obs[j] != o) ++j;
        if (j == k) { c_nodes[k] = c; c_obs[k] = o; c_score[k] = s; slot[k] = a; ++k; }
        else if (s > c_score[j]) { c_nodes[j] = c; c_score[j] = s; }
    }
    return k;
}

}  // namespace b200
