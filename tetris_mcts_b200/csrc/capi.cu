// capi.cu — host side of libb200_tetris_mcts.so: the C-ABI declared in include/b200_tetris_mcts.h.
// One engine = one CUDA stream + the per-game arenas in HBM.  No CPU compute path exists in this file: every
// entry point either launches kernels or moves bytes.
#include <cuda_runtime.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200_tetris_mcts.h"
#include "kernels.cuh"
#include "valuenet_simt.cuh"
#include "dist_dev.cuh"
#include "distnet_simt.cuh"
#include "replay_policy.cuh"
#include "valuenet_tc.cuh"
#include "distnet_tc.cuh"

using namespace b200;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t _e = (call);                                                                      \
        if (_e != cudaSuccess)                                                                        \
            return fail(B200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));           \
    } while (0)

extern "C" const char *b200_last_error(void) { return g_err.c_str(); }
extern "C" int b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

enum { PH_SELECT = 0, PH_CONV, PH_FC, PH_BACKUP, PH_ROLLOUT, PH_SYNTH, PH_MISC, PH_GC, PH_N = 8 };

struct b200_engine {
    b200_config cfg;
    Arena A;
    cudaStream_t stream = nullptr; bool own_stream = true;   // own_stream false: the caller's stream (b200_engine_set_stream), never destroyed here
    std::vector<void *> allocs;
    uint32_t *d_default_rec = nullptr;
    float *d_stats = nullptr; int32_t *d_action = nullptr;
    unsigned long long *d_game_stats = nullptr;
    // network
    bool have_weights = false;
    float *d_wraw = nullptr;
    NetWeights W{};
    float *d_act3 = nullptr; size_t act3_rows = 0;                                            // CUDA-core path
    uint8_t *d_tcw = nullptr; TcWeights TW{}; uint8_t *d_act3_tc = nullptr; size_t act3_tiles = 0;    // tensor-core path
    bool have_dist_weights = false; float *d_dnw = nullptr; DistNetWeights DW{}; float *d_dn_act = nullptr; size_t dn_rows = 0;
    uint8_t *d_dn_tcw = nullptr; DnTcWeights DTW{}; uint8_t *d_dn_act_tc = nullptr; size_t dn_act_tiles = 0;
    int n_sm = 148;
    // timing
    bool timing = false;
    std::vector<cudaEvent_t> ev; size_t ev_used = 0;
    std::vector<int> ev_phase;
    float phase_ms[PH_N] = {0}; uint64_t phase_launches[PH_N] = {0};
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    // sampling
    uint8_t *d_samples = nullptr; int sample_cap = 0; int32_t *d_sample_count = nullptr;
    // replay-memory policy (agent.cpp:619-775)
    ReplayPolicy rp; uint8_t *d_rp_tmp = nullptr, *d_rp_keep = nullptr; float *d_rp_vis = nullptr; int32_t *d_rp_kept = nullptr; int replay_alloc = 0;
    // one simulation step captured as a CUDA graph (replayed when phase timing is off: ~7 launches + 1 memset per step, 500 steps/move)
    int gc_headroom = 0;           // b200_set_gc_headroom: collect between moves every game with fewer free slots than this
    int4 *d_pc = nullptr; int32_t *d_pc_var = nullptr, *d_pc_len = nullptr; uint4 *d_pc_sib = nullptr; int4 *d_pc_own = nullptr;   // path cache (b200_set_path_cache): allocated at the first switch-on, A.pc == nullptr while off
    cudaGraphExec_t step_exec = nullptr; bool step_graph_failed = false;
    uint64_t step_launches[PH_N] = {0};
};

// kernel arguments of the captured step changed (weights, replay memory, ...): capture again at the next run_sims
static void drop_step_graph(b200_engine *e) {
    if (e->step_exec) { cudaStreamSynchronize(e->stream); cudaGraphExecDestroy(e->step_exec); e->step_exec = nullptr; }
    e->step_graph_failed = false;
}

static inline int blocks_groups(int G) { return (G + GROUPS_PER_BLOCK - 1) / GROUPS_PER_BLOCK; }
static inline int gc_blocks(const b200_engine *e) { int b = e->n_sm * 4; return e->A.G < b ? e->A.G : b; }   // k_gc CTAs (one scratch set each)

// k_backup's per-warp bitmap of the trace's observations (path cache on): max_nodes bits, four warps per CTA
static inline int backup_bitmap_words(const Arena &A) { return A.pc ? (A.M + 31) / 32 : 0; }
static inline size_t backup_smem(const Arena &A) { return (size_t)4 * backup_bitmap_words(A) * sizeof(unsigned); }

// temporary device buffers of the standalone entry points: freed on every return path
struct Scratch {
    std::vector<void *> bufs;
    ~Scratch() { for (void *q : bufs) cudaFree(q); }
    template <typename T> cudaError_t get(T **out, size_t bytes) {
        void *q = nullptr;
        cudaError_t err = cudaMalloc(&q, bytes ? bytes : 1);
        if (err == cudaSuccess) { bufs.push_back(q); *out = (T *)q; }
        return err;
    }
};

static void dfree(b200_engine *e, void *p) {   // release one engine-owned allocation early (a buffer that is being replaced)
    if (!p) return;
    for (size_t i = 0; i < e->allocs.size(); ++i)
        if (e->allocs[i] == p) { e->allocs.erase(e->allocs.begin() + i); break; }
    cudaFree(p);
}

template <typename T>
static int dalloc(b200_engine *e, T **p, size_t n, bool zero = true) {
    void *q = nullptr;
    cudaError_t err = cudaMalloc(&q, n * sizeof(T));
    if (err != cudaSuccess) return fail(B200_ERR_CUDA, std::string("cudaMalloc ") + std::to_string(n * sizeof(T)) + " B: " + cudaGetErrorString(err));
    if (zero) cudaMemsetAsync(q, 0, n * sizeof(T), e->stream);
    e->allocs.push_back(q);
    *p = (T *)q;
    return 0;
}

// SPEC §2-4 fresh games, produced ON THE DEVICE so that no host restatement of the env exists in this library.
// seeds == nullptr: every game gets the default seed (SPEC §4); reset != 0: SPEC §4 reset() of the records in place.
__global__ void k_new_games(uint32_t *recs, int n, int app, int scoring, int randomizer, const uint32_t *seeds, int reset) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Game g;
    uint32_t w[REC_WORDS];
    if (reset) {
        load_rec(recs + (size_t)i * REC_WORDS, w);
        unpack(g, w);
        reset_game(g);
    } else {
        for (int q = 0; q < 10; ++q) g.w[q] = 0;
        g.piece = 0; g.rot = 0; g.px = 3; g.py = 0; g.bag = 0x7fu; g.dropcnt = 0; g.end = 0;
        g.app = app < 1 ? 1 : (app > 255 ? 255 : app); g.scoring = scoring ? 1 : 0; g.randomizer = randomizer ? 1 : 0;
        uint32_t seed = seeds ? seeds[i] : 0u;
        g.combo = 0; g.rng = seed ? seed : 0x9E3779B9u; g.score = 0; g.lines = 0;
        for (int q = 0; q < 4; ++q) g.ls[q] = 0;
        spawn(g);
    }
    pack(g, w);
    store_rec(recs + (size_t)i * REC_WORDS, w);
}

struct PhaseTimer {
    b200_engine *e; int ph;
    PhaseTimer(b200_engine *e_, int ph_) : e(e_), ph(ph_) {
        e->phase_launches[ph] += 1;
        if (!e->timing) return;
        if (e->ev_used + 2 > e->ev.size()) {
            size_t old = e->ev.size();
            e->ev.resize(old + 4096);
            for (size_t i = old; i < e->ev.size(); ++i) cudaEventCreate(&e->ev[i]);
        }
        cudaEventRecord(e->ev[e->ev_used], e->stream);
    }
    ~PhaseTimer() {
        if (!e->timing) return;
        cudaEventRecord(e->ev[e->ev_used + 1], e->stream);
        e->ev_phase.push_back(ph);
        e->ev_used += 2;
    }
};

static void flush_timing(b200_engine *e) {
    if (!e->timing || e->ev_used == 0) return;
    cudaStreamSynchronize(e->stream);
    for (size_t i = 0; i < e->ev_used; i += 2) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e->ev[i], e->ev[i + 1]);
        e->phase_ms[e->ev_phase[i / 2]] += ms;
    }
    e->ev_used = 0; e->ev_phase.clear();
}

extern "C" int b200_engine_create(const b200_config *cfg, b200_engine **out) {
    if (!cfg || !out) return fail(B200_ERR_BAD_ARG, "null argument");
    if (cfg->n_games < 1 || cfg->max_nodes < 16 || cfg->max_nodes >= (1 << 28) || (cfg->max_nodes & 3))
        return fail(B200_ERR_BAD_ARG, "n_games >= 1, 16 <= max_nodes < 2^28, max_nodes % 4 == 0");
    if (cfg->mode < 0 || cfg->mode > 3) return fail(B200_ERR_BAD_ARG, "mode");
    if (cfg->mode == MODE_DIST && (cfg->dist_bins < 2 || cfg->dist_bins > 64 || !(cfg->dist_vmax > cfg->dist_vmin)))
        return fail(B200_ERR_BAD_ARG, "distributional mode needs 2 <= dist_bins <= 64 and dist_vmax > dist_vmin");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    CK(cudaSetDevice(cfg->device));
    b200_engine *e = new b200_engine();
    struct Guard { b200_engine *e; ~Guard() { if (e) b200_engine_destroy(e); } } guard{e};   // every failing return below destroys the half-built engine
    e->cfg = *cfg;
    CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, cfg->device));
    e->n_sm = prop.multiProcessorCount;
    Arena &A = e->A;
    memset(&A, 0, sizeof(A));
    A.G = cfg->n_games; A.M = cfg->max_nodes;
    int H = A.M + A.M / 2;                       // load factor <= 2/3 (tombstones only live inside k_gc, which rebuilds both tables)
    if (H < 16) H = 16;
    A.H = H; A.trace_max = cfg->trace_max > 0 ? cfg->trace_max : 512;
    A.mode = cfg->mode; A.low = cfg->low; A.lp_end_from_obs = cfg->lp_end_from_obs; A.lp_var_gamma2 = cfg->lp_var_gamma2;
    A.stale_pop = cfg->stale_pop; A.eval_kind = cfg->eval_kind; A.overflow_reset = cfg->overflow_reset; A.gc_min_gain = cfg->overflow_reset ? cfg->max_nodes / 8 : 0; A.gamma = cfg->gamma; A.rollout_variance = cfg->rollout_variance;
    size_t GM = (size_t)A.G * A.M, G = (size_t)A.G;
    int rc = 0;
    rc |= dalloc(e, &A.row, GM * ROW_WORDS);
    rc |= dalloc(e, &A.stat, GM);
    rc |= dalloc(e, &A.rec, GM * REC_WORDS, false);
    rc |= dalloc(e, &A.key, GM * KEY_WORDS);
    rc |= dalloc(e, &A.ntab, G * H);
    rc |= dalloc(e, &A.otab, G * H);
    rc |= dalloc(e, &A.nfree, GM); rc |= dalloc(e, &A.ofree, GM);
    rc |= dalloc(e, &A.n_nfree, G); rc |= dalloc(e, &A.n_ofree, G);
    rc |= dalloc(e, &A.root, G); rc |= dalloc(e, &A.episode, G); rc |= dalloc(e, &A.status, G); rc |= dalloc(e, &A.srng, G);
    rc |= dalloc(e, &A.trace, G * A.trace_max); rc |= dalloc(e, &A.trace_len, G); rc |= dalloc(e, &A.leaf_kind, G);
    rc |= dalloc(e, &A.trace_meta, G * A.trace_max);
    {   // collection scratch: one set per k_gc CTA (gc_blocks), not per game
        const size_t pool = (size_t)gc_blocks(e) * A.M;
        rc |= dalloc(e, &A.nmark, pool); rc |= dalloc(e, &A.omark, pool); rc |= dalloc(e, &A.gc_queue, pool * 2);
    }
    rc |= dalloc(e, &A.cur, G * REC_WORDS);
    rc |= dalloc(e, &A.req, G * 8); rc |= dalloc(e, &A.n_req, 2);
    rc |= dalloc(e, &A.gc_list, G); rc |= dalloc(e, &A.pending, G); rc |= dalloc(e, &A.resume_a, G);
    rc |= dalloc(e, &A.eval_out, G * 8); rc |= dalloc(e, &A.rollout_val, G);
    rc |= dalloc(e, &A.counters, 48);
    A.fin_cap = 4 * A.G;
    rc |= dalloc(e, &A.fin_log, (size_t)A.fin_cap * 4); rc |= dalloc(e, &A.fin_count, 1);
    if (cfg->mode == MODE_DIST) {
        A.dist_bins = cfg->dist_bins; A.dist_vmin = cfg->dist_vmin; A.dist_vmax = cfg->dist_vmax;
        rc |= dalloc(e, &A.nstat, GM * NSTAT_WORDS); rc |= dalloc(e, &A.ndist, GM * (size_t)A.dist_bins); rc |= dalloc(e, &A.dist_eval, G * (size_t)A.dist_bins);
    }
    rc |= dalloc(e, &e->d_default_rec, REC_WORDS);
    rc |= dalloc(e, &e->d_stats, G * 21); rc |= dalloc(e, &e->d_action, G);
    e->d_game_stats = A.counters + 8;
    float *zt = nullptr;
    rc |= dalloc(e, &zt, ZTABLE_N);
    if (rc) return B200_ERR_CUDA;
    {   // z(n) = norm_quantile(n) narrowed to float: special.h:26-33 + core.h:93, evaluated with the host libm
        std::vector<float> h(ZTABLE_N);
        const double l2 = log(2.0), l22 = log(22.0), l41 = log(41.0);
        for (int n = 0; n < ZTABLE_N; ++n) {
            double t = (double)n, alpha = 1 - 1 / t;
            h[n] = (float)(10 * log(1 - log(-log(alpha) / l2) / l22) / l41);
        }
        CK(cudaMemcpyAsync(zt, h.data(), ZTABLE_N * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        A.ztable = zt;
    }
    k_new_games<<<1, 1, 0, e->stream>>>(e->d_default_rec, 1, cfg->actions_per_drop, cfg->scoring, cfg->randomizer, nullptr, 0);
    k_init_arena<<<e->n_sm * 8, 256, 0, e->stream>>>(A, e->d_default_rec, cfg->seed);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    guard.e = nullptr;
    *out = e;
    return B200_OK;
}

extern "C" int b200_engine_destroy(b200_engine *e) {
    if (!e) return B200_OK;
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->step_exec) cudaGraphExecDestroy(e->step_exec);
    for (void *p : e->allocs) cudaFree(p);
    for (auto &ev : e->ev) cudaEventDestroy(ev);
    if (e->t0) { cudaEventDestroy(e->t0); cudaEventDestroy(e->t1); }
    if (e->stream && e->own_stream) cudaStreamDestroy(e->stream);
    delete e;
    return B200_OK;
}

// SURVEY 8(b).5 "explicit cudaStream_t": all work of the engine is issued on `cuda_stream` from now on (nullptr: a private non-blocking
// stream again).  The engine drains its current stream first, so nothing of it is in flight on two streams at once; the captured
// simulation step is dropped and re-captured on the new stream.  The caller keeps ownership of its stream and must keep it alive.
extern "C" int b200_engine_set_stream(b200_engine *e, void *cuda_stream) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    drop_step_graph(e);
    cudaStream_t ns = (cudaStream_t)cuda_stream;
    const bool own = ns == nullptr;
    if (own) CK(cudaStreamCreateWithFlags(&ns, cudaStreamNonBlocking));
    if (e->own_stream) cudaStreamDestroy(e->stream);
    e->stream = ns; e->own_stream = own;
    return B200_OK;
}

extern "C" int b200_engine_get_stream(b200_engine *e, void **cuda_stream_out) {
    if (!e || !cuda_stream_out) return fail(B200_ERR_BAD_ARG, "null argument");
    *cuda_stream_out = (void *)e->stream;
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- weights
extern "C" int b200_load_weights(b200_engine *e, const float *w) {
    if (!e || !w) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    const float *c1w = w, *c1b = c1w + 288, *c2w = c1b + 32, *c2b = c2w + 9216, *c3w = c2b + 32, *c3b = c3w + 9216;
    const float *f1w = c3b + 32, *f1b = f1w + 458752, *fow = f1b + 256, *fob = fow + 512, *ub = fob + 2, *lb = ub + 2;
    // pure re-layout (no arithmetic): see NetWeights
    std::vector<float> h;
    h.resize(288 + 9216 * 2 + 96 + (size_t)1792 * 256 + 256 + 512 + 6);
    float *p = h.data();
    float *w1 = p; p += 288;
    float *w2 = p; p += 9216;
    float *w3 = p; p += 9216;
    float *b123 = p; p += 96;
    float *wf = p; p += (size_t)1792 * 256;
    float *bf = p; p += 256;
    float *wo = p; p += 512;
    float *tail = p;
    for (int co = 0; co < 32; ++co)
        for (int tap = 0; tap < 9; ++tap) w1[tap * 32 + co] = c1w[co * 9 + tap];
    for (int co = 0; co < 32; ++co)
        for (int ci = 0; ci < 32; ++ci)
            for (int tap = 0; tap < 9; ++tap) {
                w2[(ci * 9 + tap) * 32 + co] = c2w[(co * 32 + ci) * 9 + tap];
                w3[(ci * 9 + tap) * 32 + co] = c3w[(co * 32 + ci) * 9 + tap];
            }
    memcpy(b123, c1b, 128); memcpy(b123 + 32, c2b, 128); memcpy(b123 + 64, c3b, 128);
    for (int n = 0; n < 256; ++n)
        for (int c = 0; c < 32; ++c)
            for (int y = 0; y < 14; ++y)
                for (int x = 0; x < 4; ++x) wf[(size_t)((y * 32 + c) * 4 + x) * 256 + n] = f1w[(size_t)n * 1792 + c * 56 + y * 4 + x];
    memcpy(bf, f1b, 1024); memcpy(wo, fow, 2048);
    tail[0] = fob[0]; tail[1] = fob[1]; tail[2] = ub[0]; tail[3] = ub[1]; tail[4] = lb[0]; tail[5] = lb[1];
    if (!e->d_wraw) { if (dalloc(e, &e->d_wraw, h.size(), false)) return B200_ERR_CUDA; }
    CK(cudaMemcpyAsync(e->d_wraw, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    float *d = e->d_wraw;
    e->W.w1 = d; e->W.w2 = d + 288; e->W.w3 = d + 288 + 9216; e->W.b1 = d + 288 + 18432; e->W.b2 = e->W.b1 + 32; e->W.b3 = e->W.b1 + 64;
    e->W.wfc1 = e->W.b1 + 96; e->W.bfc1 = e->W.wfc1 + (size_t)1792 * 256; e->W.wout = e->W.bfc1 + 256;
    e->W.bout = e->W.wout + 512; e->W.ub = e->W.bout + 2; e->W.lb = e->W.bout + 4;
    CK(cudaFuncSetAttribute(k_vn_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, VN_SMEM_BYTES));
    if (!e->d_tcw && dalloc(e, &e->d_tcw, TC_PACKED_BYTES, false)) return B200_ERR_CUDA;
    if (tc_prepare(w, e->d_tcw, e->TW, e->stream)) return fail(B200_ERR_CUDA, "tensor-core weight preparation failed");
    e->have_weights = true;
    drop_step_graph(e);
    return B200_OK;
}

// Grow a network's activation buffer to `need` units of `unit` elements.  A replaced buffer (a larger standalone batch) is only freed once
// the stream has drained, and the captured step graph, which holds its address, is dropped.
template <typename T>
static int grow_act(b200_engine *e, T **buf, size_t *have, size_t need, size_t unit, bool zero) {
    if (*have >= need) return 0;
    const bool moved = *buf != nullptr;
    if (moved) { cudaStreamSynchronize(e->stream); dfree(e, *buf); *buf = nullptr; *have = 0; }
    if (dalloc(e, buf, need * unit, zero)) return B200_ERR_CUDA;
    *have = need;
    if (moved) drop_step_graph(e);
    return 0;
}
static inline size_t tiles_of(size_t rows) { return (rows + 127) / 128; }

// run the network over the request list req[0..*n_req) -> eval_out; device-side count, no host sync
static int launch_net(b200_engine *e, const uint2 *req, const int32_t *n_req, const uint32_t *keys, int M, float2 *eval_out,
                      size_t max_rows) {
    if (!e->have_weights) return fail(B200_ERR_NO_WEIGHTS, "b200_load_weights was not called");
    if (e->cfg.eval_kind == B200_EVAL_NET_TC) {
        if (grow_act(e, &e->d_act3_tc, &e->act3_tiles, tiles_of(max_rows), TcfPipe::ACT_TILE_BYTES, true)) return B200_ERR_CUDA;
        {
            PhaseTimer t(e, PH_CONV);
            k_tc_conv<<<e->n_sm, TCC_THREADS, TCC_SMEM, e->stream>>>(e->W, e->TW, req, n_req, keys, M, e->d_act3_tc, (int)e->act3_tiles,
                                                                    e->timing ? e->A.counters + 16 : nullptr);
        }
        {
            PhaseTimer t(e, PH_FC);
            k_tc_fc<<<e->n_sm, FC_PIPE_THREADS, TCF_SMEM, e->stream>>>(e->W, e->TW, e->d_act3_tc, (int)e->act3_tiles, req, n_req, eval_out);
        }
        CK(cudaGetLastError());
        return B200_OK;
    }
    if (grow_act(e, &e->d_act3, &e->act3_rows, max_rows, 1792, false)) return B200_ERR_CUDA;
    {
        PhaseTimer t(e, PH_CONV);
        k_vn_conv<<<e->n_sm, VN_THREADS, VN_SMEM_BYTES, e->stream>>>(e->W, req, n_req, keys, M, e->d_act3);
    }
    {
        PhaseTimer t(e, PH_FC);
        k_vn_fc<<<e->n_sm * 2, FC_THREADS, 0, e->stream>>>(e->W, e->d_act3, req, n_req, eval_out);
    }
    CK(cudaGetLastError());
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- distributional network
__global__ void k_states_to_keys(const int8_t *states, int k, uint32_t *keys, uint2 *req);   // defined with the standalone value net below

// standalone forward: k boards -> device keys and one request per board (buffers of `rows` >= k entries), request count k on the device
static int stage_boards(b200_engine *e, Scratch &tmp, const int8_t *states, int k, size_t rows, uint32_t **d_keys, uint2 **d_req, int32_t **d_n) {
    int8_t *d_states = nullptr;
    CK(tmp.get(&d_states, (size_t)k * 200)); CK(tmp.get(d_keys, rows * KEY_WORDS * 4)); CK(tmp.get(d_req, rows * 8)); CK(tmp.get(d_n, 4));
    CK(cudaMemcpyAsync(d_states, states, (size_t)k * 200, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(*d_n, &k, 4, cudaMemcpyHostToDevice, e->stream));
    k_states_to_keys<<<(k + 127) / 128, 128, 0, e->stream>>>(d_states, k, *d_keys, *d_req);
    return B200_OK;
}

extern "C" int b200_load_dist_weights(b200_engine *e, const float *w, int atoms) {
    if (!e || !w || atoms < 2 || atoms > 64) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    if (e->A.mode == MODE_DIST && atoms != e->A.dist_bins) return fail(B200_ERR_BAD_ARG, "atoms must equal dist_bins");
    std::vector<float> h;
    dn_relayout(w, atoms, h);
    if (!e->d_dnw) { if (dalloc(e, &e->d_dnw, h.size(), false)) return B200_ERR_CUDA; }
    CK(cudaMemcpyAsync(e->d_dnw, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->DW = dn_pointers(e->d_dnw, atoms);
    CK(cudaFuncSetAttribute(k_dn_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, DN_CONV_SMEM));
    CK(cudaFuncSetAttribute(k_dn_fc, cudaFuncAttributeMaxDynamicSharedMemorySize, DN_FC_SMEM));
    if (!e->d_dn_tcw && dalloc(e, &e->d_dn_tcw, DN_TC_PACKED_BYTES, false)) return B200_ERR_CUDA;
    if (dn_tc_prepare(w, e->d_dn_tcw, e->DTW, e->stream)) return fail(B200_ERR_CUDA, "tensor-core weight preparation (distributional network) failed");
    e->have_dist_weights = true;
    drop_step_graph(e);
    return B200_OK;
}

static int launch_distnet_on(b200_engine *e, const uint2 *req, const int32_t *n_req, const uint32_t *keys, int M, float *out, size_t max_rows) {
    if (!e->have_dist_weights) return fail(B200_ERR_NO_WEIGHTS, "b200_load_dist_weights was not called");
    if (e->cfg.eval_kind == B200_EVAL_NET_TC) {
        if (grow_act(e, &e->d_dn_act_tc, &e->dn_act_tiles, tiles_of(max_rows), TdfPipe::ACT_TILE_BYTES, true)) return B200_ERR_CUDA;
        {
            PhaseTimer t(e, PH_CONV);
            k_tdc_conv<<<e->n_sm, TDC_THREADS, TDC_SMEM, e->stream>>>(e->DW, e->DTW, req, n_req, keys, M, e->d_dn_act_tc, (int)e->dn_act_tiles);
        }
        {
            PhaseTimer t(e, PH_FC);
            k_tdc_fc<<<e->n_sm, FC_PIPE_THREADS, TDF_SMEM, e->stream>>>(e->DW, e->DTW, e->d_dn_act_tc, (int)e->dn_act_tiles, req, n_req, out);
        }
        CK(cudaGetLastError());
        return B200_OK;
    }
    if (grow_act(e, &e->d_dn_act, &e->dn_rows, max_rows, 2048, false)) return B200_ERR_CUDA;
    {
        PhaseTimer t(e, PH_CONV);
        k_dn_conv<<<e->n_sm * 2, DN_THREADS, DN_CONV_SMEM, e->stream>>>(e->DW, req, n_req, keys, M, e->d_dn_act);
    }
    {
        PhaseTimer t(e, PH_FC);
        k_dn_fc<<<e->n_sm, DN_THREADS, DN_FC_SMEM, e->stream>>>(e->DW, e->d_dn_act, req, n_req, out);
    }
    CK(cudaGetLastError());
    return B200_OK;
}
static int launch_distnet(b200_engine *e) {
    return launch_distnet_on(e, e->A.req, e->A.n_req, e->A.key, e->A.M, e->A.dist_eval, (size_t)e->A.G);
}

// Model.inference of model/model_distributional.py (softmax over atoms): states[k][200] int8 -> dist[k][atoms]
extern "C" int b200_distnet_forward(b200_engine *e, const int8_t *states, int k, int atoms, float *dist) {
    if (!e || !states || !dist || k < 1 || atoms != e->DW.atoms) return fail(B200_ERR_BAD_ARG, "bad argument (atoms must match the loaded weights)");
    CK(cudaSetDevice(e->cfg.device));
    uint32_t *d_keys = nullptr; uint2 *d_req = nullptr; int32_t *d_n = nullptr; float *d_out = nullptr;
    Scratch tmp;
    if (int rc = stage_boards(e, tmp, states, k, (size_t)k, &d_keys, &d_req, &d_n)) return rc;
    CK(tmp.get(&d_out, (size_t)k * atoms * 4));
    k_dn_req_rows<<<(k + 127) / 128, 128, 0, e->stream>>>(d_req, k);      // request i -> output row i
    int rc = launch_distnet_on(e, d_req, d_n, d_keys, 0, d_out, (size_t)k);
    if (rc == B200_OK) {
        cudaError_t ce = cudaMemcpyAsync(dist, d_out, (size_t)k * atoms * 4, cudaMemcpyDeviceToHost, e->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
        if (ce != cudaSuccess) rc = fail(B200_ERR_CUDA, cudaGetErrorString(ce));
    }
    cudaStreamSynchronize(e->stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------------- games / roots

static int check_status(b200_engine *e) {   // cheap: max over the status array computed on the host after a small copy
    std::vector<int32_t> st(e->A.G);
    CK(cudaMemcpyAsync(st.data(), e->A.status, st.size() * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int g = 0; g < e->A.G; ++g)
        if (st[g] != ST_OK && !((st[g] == ST_ARENA_FULL || st[g] == ST_RESET_DONE) && e->A.overflow_reset)) {
            int code = st[g] == ST_ARENA_FULL ? B200_ERR_ARENA_FULL : B200_ERR_TRACE_FULL;
            return fail(code, "game " + std::to_string(g) + (st[g] == ST_ARENA_FULL ? ": arena full after garbage collection (raise max_nodes)" : ": trace longer than trace_max"));
        }
    return B200_OK;
}

// TreeAgent.remove_nodes() (agents/agent.py:246-257) for every game with fewer than min_free free node slots, as ONE batched k_gc
extern "C" int b200_remove_nodes(b200_engine *e, int min_free) {
    if (!e || min_free < 0) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    {
        PhaseTimer t(e, PH_GC);
        CK(cudaMemsetAsync(e->A.n_req + 1, 0, sizeof(int32_t), e->stream));
        k_gc_request<<<(e->A.G + 127) / 128, 128, 0, e->stream>>>(e->A, min_free);
        k_gc<<<gc_blocks(e), GC_THREADS, 0, e->stream>>>(e->A);
    }
    CK(cudaGetLastError());
    return B200_OK;
}

extern "C" int b200_set_gc_headroom(b200_engine *e, int min_free) {
    if (!e || min_free < 0) return fail(B200_ERR_BAD_ARG, "bad argument");
    e->gc_headroom = min_free;
    return B200_OK;
}

// Path cache (search_dev.cuh "path cache"): scheduling/memory-traffic only, no effect on any result.  LP mode, max_nodes <= 65536.
extern "C" int b200_set_path_cache(b200_engine *e, int on) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    if (on) {
        if (e->A.mode != MODE_LP) return fail(B200_ERR_BAD_ARG, "the path cache serves B200_MODE_LP (its coherence rules rest on the LP backup)");
        if (e->A.M > PC_MAX_NODES) return fail(B200_ERR_BAD_ARG, "the path cache needs max_nodes <= 65536 (k_backup's bitmap of the trace's observations)");
    }
    CK(cudaStreamSynchronize(e->stream));
    drop_step_graph(e);
    if (on && !e->d_pc) {
        const size_t levels = (size_t)e->A.G * e->A.trace_max;
        if (dalloc(e, &e->d_pc, levels * 8, false) || dalloc(e, &e->d_pc_var, levels * 8, false) || dalloc(e, &e->d_pc_sib, levels, false) || dalloc(e, &e->d_pc_own, levels, false) ||
            dalloc(e, &e->d_pc_len, (size_t)e->A.G)) return B200_ERR_CUDA;
    }
    if (on) CK(cudaMemsetAsync(e->d_pc_len, 0, (size_t)e->A.G * sizeof(int32_t), e->stream));   // nothing is valid until a walk has left its entries
    e->A.pc = on ? e->d_pc : nullptr;
    e->A.pc_var = on ? e->d_pc_var : nullptr;
    e->A.pc_len = on ? e->d_pc_len : nullptr;
    e->A.pc_sib = on ? e->d_pc_sib : nullptr;
    e->A.pc_own = on ? e->d_pc_own : nullptr;
    return B200_OK;
}

static int update_root_impl(b200_engine *e, int auto_reset, bool headroom_collection) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    {
        PhaseTimer t(e, PH_MISC);
        CK(cudaMemsetAsync(e->A.n_req + 1, 0, sizeof(int32_t), e->stream));
        k_update_root<<<blocks_groups(e->A.G), TPB, 0, e->stream>>>(e->A, auto_reset, e->d_game_stats, 0);
        k_gc<<<gc_blocks(e), GC_THREADS, 0, e->stream>>>(e->A);                 // games whose free list ran dry (usually none)
        k_update_root<<<blocks_groups(e->A.G), TPB, 0, e->stream>>>(e->A, auto_reset, e->d_game_stats, 1);
    }
    if (headroom_collection && e->gc_headroom > 0) {
        int rc = b200_remove_nodes(e, e->gc_headroom);
        if (rc) return rc;
    }
    CK(cudaGetLastError());
    return B200_OK;
}

extern "C" int b200_update_root(b200_engine *e, int auto_reset) { return update_root_impl(e, auto_reset, true); }

extern "C" int b200_set_games(b200_engine *e, const uint32_t *recs) {
    if (!e || !recs) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(e->A.cur, recs, (size_t)e->A.G * REC_WORDS * 4, cudaMemcpyHostToDevice, e->stream));
    int rc = update_root_impl(e, 0, false);   // handing the games over is not a move: the driver's between-moves collection (b200_set_gc_headroom) is not due here
    if (rc) return rc;
    return check_status(e);
}

extern "C" int b200_get_games(b200_engine *e, uint32_t *recs) {
    if (!e || !recs) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(recs, e->A.cur, (size_t)e->A.G * REC_WORDS * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- simulations
// One simulation step of every game: select+expand -> (collect garbage, resume) -> evaluate -> backup.
static int enqueue_step(b200_engine *e) {
    const Arena &A = e->A;
    const int G = A.G;
    CK(cudaMemsetAsync(A.n_req, 0, 2 * sizeof(int32_t), e->stream));
    {
        PhaseTimer t(e, PH_SELECT);
        Arena Ap = A;
        Ap.prof = e->timing ? A.counters + 32 : nullptr;
        k_select_expand<<<(G + SE_GAMES_PER_BLOCK - 1) / SE_GAMES_PER_BLOCK, TPB, 0, e->stream>>>(Ap);
    }
    {   // remove_nodes for the games that ran out of free slots in this step, then the rest of their expansion
        PhaseTimer t(e, PH_GC);
        k_gc<<<gc_blocks(e), GC_THREADS, 0, e->stream>>>(A);
        k_expand_resume<<<blocks_groups(G), TPB, 0, e->stream>>>(A);
    }
    if (A.mode == MODE_VANILLA) {
        PhaseTimer t(e, PH_ROLLOUT);
        k_rollout<<<(G + 63) / 64, 64, 0, e->stream>>>(A);
    } else if (A.mode == MODE_DIST) {
        if (e->cfg.eval_kind == B200_EVAL_SYNTHETIC) {
            PhaseTimer t(e, PH_SYNTH);
            k_eval_synthetic_dist<<<(G + 127) / 128, 128, 0, e->stream>>>(A);
        } else {
            int rc = launch_distnet(e);
            if (rc) return rc;
        }
    } else if (e->cfg.eval_kind == B200_EVAL_SYNTHETIC) {
        PhaseTimer t(e, PH_SYNTH);
        k_eval_synthetic<<<(G * 7 + 255) / 256 < 1184 ? (G * 7 + 255) / 256 : 1184, 256, 0, e->stream>>>(A);
    } else {
        int rc = launch_net(e, A.req, A.n_req, A.key, A.M, A.eval_out, (size_t)G * (A.mode == MODE_LP ? 7 : 1));
        if (rc) return rc;
    }
    {
        PhaseTimer t(e, PH_BACKUP);
        if (A.mode == MODE_DIST) k_dist_backup<<<(G + 3) / 4, 128, 0, e->stream>>>(A);
        else k_backup<<<(G + 3) / 4, 128, backup_smem(A), e->stream>>>(A, backup_bitmap_words(A));
    }
    return B200_OK;
}

// Capture one step (same launches, same arguments every step: all sizes are read on the device) and replay it.  The first
// step of an engine runs directly so that lazily allocated buffers (activations) exist before the capture.
static void capture_step(b200_engine *e) {
    uint64_t before[PH_N];
    for (int i = 0; i < PH_N; ++i) before[i] = e->phase_launches[i];
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); e->step_graph_failed = true; return; }
    int rc = enqueue_step(e);
    cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
    for (int i = 0; i < PH_N; ++i) { e->step_launches[i] = e->phase_launches[i] - before[i]; e->phase_launches[i] = before[i]; }
    if (rc == B200_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&e->step_exec, graph, 0) == cudaSuccess) {
        cudaGraphDestroy(graph);
        return;
    }
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    e->step_exec = nullptr; e->step_graph_failed = true;    // direct launches from now on
}

extern "C" int b200_run_sims(b200_engine *e, int sims) {
    if (!e || sims < 0) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    const Arena &A = e->A;
    const bool need_net = A.mode != MODE_VANILLA && e->cfg.eval_kind != B200_EVAL_SYNTHETIC;
    if (need_net && !(A.mode == MODE_DIST ? e->have_dist_weights : e->have_weights)) return fail(B200_ERR_NO_WEIGHTS, "b200_load_weights was not called");
    CK(cudaMemsetAsync(A.counters + 12, 0, sizeof(unsigned long long), e->stream));   // counter 12: the longest trace of this call
    for (int s = 0; s < sims; ++s) {
        if (!e->timing && e->step_exec) {
            CK(cudaGraphLaunch(e->step_exec, e->stream));
            for (int i = 0; i < PH_N; ++i) e->phase_launches[i] += e->step_launches[i];
            continue;
        }
        int rc = enqueue_step(e);
        if (rc) return rc;
        if (!e->timing && !e->step_exec && !e->step_graph_failed) capture_step(e);
    }
    CK(cudaGetLastError());
    return B200_OK;
}

extern "C" int b200_get_stats(b200_engine *e, float *stats, int32_t *action) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    {
        PhaseTimer t(e, PH_MISC);
        k_root_stats<<<(e->A.G + 127) / 128, 128, 0, e->stream>>>(e->A, e->d_stats, e->d_action);
    }
    CK(cudaGetLastError());
    if (stats) CK(cudaMemcpyAsync(stats, e->d_stats, (size_t)e->A.G * 21 * 4, cudaMemcpyDeviceToHost, e->stream));
    if (action) CK(cudaMemcpyAsync(action, e->d_action, (size_t)e->A.G * 4, cudaMemcpyDeviceToHost, e->stream));
    return check_status(e);
}

extern "C" int b200_env_step(b200_engine *e, const int32_t *actions) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    if (actions) CK(cudaMemcpyAsync(e->d_action, actions, (size_t)e->A.G * 4, cudaMemcpyHostToDevice, e->stream));
    {
        PhaseTimer t(e, PH_MISC);
        k_env_step<<<(e->A.G + 127) / 128, 128, 0, e->stream>>>(e->A.cur, e->d_action, e->A.G);
    }
    CK(cudaGetLastError());
    return B200_OK;
}

extern "C" int b200_play_move(b200_engine *e, int sims, int auto_reset, int32_t *actions_out, float *stats_out) {
    int rc = b200_run_sims(e, sims);
    if (rc) return rc;
    rc = b200_get_stats(e, stats_out, actions_out);
    if (rc) return rc;
    rc = b200_env_step(e, nullptr);
    if (rc) return rc;
    rc = b200_update_root(e, auto_reset);
    if (rc) return rc;
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// The episodes that ended (and were reset) in the update_root calls since the last drain: out4[i] = {game, score, line_clears, episode},
// at most `cap` rows, count_out = how many ended (may exceed cap: the log holds 4 * n_games rows between drains).  play.py:161-177.
extern "C" int b200_finished_games(b200_engine *e, int32_t *out4, int cap, int32_t *count_out) {
    if (!e || !out4 || cap < 0 || !count_out) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    int32_t n = 0;
    CK(cudaMemcpyAsync(&n, e->A.fin_count, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    *count_out = n;
    int m = n < e->A.fin_cap ? n : e->A.fin_cap;
    if (m > cap) m = cap;
    if (m > 0) CK(cudaMemcpyAsync(out4, e->A.fin_log, (size_t)m * 16, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemsetAsync(e->A.fin_count, 0, 4, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

extern "C" int b200_status(b200_engine *e, int32_t *status) {
    if (!e || !status) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(status, e->A.status, (size_t)e->A.G * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int g = 0; g < e->A.G; ++g)
        status[g] = (status[g] == ST_OK || status[g] == ST_RESET_DONE) ? 0 : (status[g] == ST_ARENA_FULL ? B200_ERR_ARENA_FULL : B200_ERR_TRACE_FULL);
    return B200_OK;
}

extern "C" int b200_counters(b200_engine *e, uint64_t *out16) {
    if (!e || !out16) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(out16, e->A.counters, 16 * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

extern "C" int b200_debug_prof(b200_engine *e, uint64_t *out16) {   // clock64 phase sums of CTA 0 of k_tc_conv (timing mode)
    if (!e || !out16) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(out16, e->A.counters + 16, 16 * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

extern "C" int b200_debug_prof_tree(b200_engine *e, uint64_t *out16) {   // clock64 sums of sampled groups of k_select_expand (timing mode)
    if (!e || !out16) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(out16, e->A.counters + 32, 16 * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

extern "C" int b200_debug_trace_lens(b200_engine *e, int32_t *out) {   // development aid: trace length of every game's last simulation
    if (!e || !out) return fail(B200_ERR_BAD_ARG, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(out, e->A.trace_len, (size_t)e->A.G * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

extern "C" int b200_sync(b200_engine *e) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// device-side stopwatch on the engine's own stream (torch.cuda.Event only sees torch's current stream)
extern "C" int b200_timer_start(b200_engine *e) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    if (!e->t0) { CK(cudaEventCreate(&e->t0)); CK(cudaEventCreate(&e->t1)); }
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaEventRecord(e->t0, e->stream));
    return B200_OK;
}
extern "C" int b200_timer_stop(b200_engine *e, float *ms) {
    if (!e || !ms || !e->t0) return fail(B200_ERR_BAD_ARG, "timer not started");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaEventRecord(e->t1, e->stream));
    CK(cudaEventSynchronize(e->t1));
    CK(cudaEventElapsedTime(ms, e->t0, e->t1));
    return B200_OK;
}

extern "C" int b200_set_timing(b200_engine *e, int on) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    flush_timing(e);
    e->timing = on != 0;
    for (int i = 0; i < PH_N; ++i) { e->phase_ms[i] = 0; e->phase_launches[i] = 0; }
    return B200_OK;
}

extern "C" int b200_phase_ms(b200_engine *e, float *ms8, uint64_t *launches8) {
    if (!e) return fail(B200_ERR_BAD_ARG, "null engine");
    flush_timing(e);
    for (int i = 0; i < PH_N; ++i) { if (ms8) ms8[i] = e->phase_ms[i]; if (launches8) launches8[i] = e->phase_launches[i]; }
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- export
extern "C" int b200_export_game(b200_engine *e, int game, int32_t *child, float *score, int32_t *episode, int32_t *n2o,
                                int32_t *visit, float *value, float *variance, uint8_t *obs_end, uint32_t *game_recs,
                                uint32_t *obs_keys, int32_t *root, int32_t *last_trace, int32_t *last_trace_len) {
    if (!e || game < 0 || game >= e->A.G) return fail(B200_ERR_BAD_ARG, "bad game index");
    CK(cudaSetDevice(e->cfg.device));
    const Arena &A = e->A;
    size_t M = A.M;
    std::vector<int32_t> row(M * ROW_WORDS);
    std::vector<int4> stat(M);
    CK(cudaMemcpyAsync(row.data(), A.row + (size_t)game * M * ROW_WORDS, row.size() * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(stat.data(), A.stat + (size_t)game * M, M * sizeof(int4), cudaMemcpyDeviceToHost, e->stream));
    if (game_recs) CK(cudaMemcpyAsync(game_recs, A.rec + (size_t)game * M * REC_WORDS, M * REC_WORDS * 4, cudaMemcpyDeviceToHost, e->stream));
    if (obs_keys) CK(cudaMemcpyAsync(obs_keys, A.key + (size_t)game * M * KEY_WORDS, M * KEY_WORDS * 4, cudaMemcpyDeviceToHost, e->stream));
    if (root) CK(cudaMemcpyAsync(root, A.root + game, 4, cudaMemcpyDeviceToHost, e->stream));
    int32_t tl = 0;
    CK(cudaMemcpyAsync(&tl, A.trace_len + game, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (last_trace_len) *last_trace_len = tl;
    if (last_trace && tl > 0) {
        CK(cudaMemcpyAsync(last_trace, A.trace + (size_t)game * A.trace_max, (size_t)tl * 4, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
    }
    for (size_t i = 0; i < M; ++i) {   // unpack the 96-byte node record into the reference's separate arrays (agent.py:58-88)
        const int32_t *r = &row[i * ROW_WORDS];
        if (child) for (int a = 0; a < 7; ++a) child[i * 7 + a] = r[a];
        if (episode) episode[i] = r[7];
        if (n2o) n2o[i] = r[15];
        if (score) memcpy(&score[i], &r[23], 4);
        if (visit) visit[i] = stat[i].x;
        if (value) memcpy(&value[i], &stat[i].y, 4);
        if (variance) memcpy(&variance[i], &stat[i].z, 4);
        if (obs_end) obs_end[i] = (uint8_t)(stat[i].w != 0);
    }
    return B200_OK;
}

extern "C" int b200_export_dist(b200_engine *e, int game, float *node_stats, float *node_dist) {
    if (!e || game < 0 || game >= e->A.G || !e->A.nstat) return fail(B200_ERR_BAD_ARG, "not a distributional engine / bad game index");
    CK(cudaSetDevice(e->cfg.device));
    size_t M = e->A.M;
    std::vector<float> ns(M * NSTAT_WORDS);
    CK(cudaMemcpyAsync(ns.data(), e->A.nstat + (size_t)game * M * NSTAT_WORDS, ns.size() * 4, cudaMemcpyDeviceToHost, e->stream));
    if (node_dist) CK(cudaMemcpyAsync(node_dist, e->A.ndist + (size_t)game * M * e->A.dist_bins, M * e->A.dist_bins * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (node_stats) for (size_t i = 0; i < M; ++i) for (int j = 0; j < 5; ++j) node_stats[i * 5 + j] = ns[i * NSTAT_WORDS + j];
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- standalone value net
__global__ void k_states_to_keys(const int8_t *states, int k, uint32_t *keys, uint2 *req) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const int8_t *s = states + (size_t)i * 200;
    uint32_t key[KEY_WORDS];
    for (int q = 0; q < KEY_WORDS; ++q) key[q] = 0;
    uint32_t cells = 0; int n = 0;
    for (int c = 0; c < 200; ++c) {
        int r = c / 10, x = c % 10;
        if (s[c] > 0) key[r >> 1] |= 1u << ((r & 1) * 16 + x);
        else if (s[c] < 0 && n < 4) { cells |= (uint32_t)c << (8 * n); ++n; }
    }
    for (; n < 4; ++n) cells |= 0xffu << (8 * n);   // fewer than four -1 cells: no such cell index (255)
    key[10] = cells;
    for (int q = 0; q < KEY_WORDS; ++q) keys[(size_t)i * KEY_WORDS + q] = key[q];
    // every standalone request gets its own output slot: game = i/8, slot = i%8 -> eval_out[i]
    req[i] = make_uint2((uint32_t)(i >> 3), (uint32_t)i | ((uint32_t)(i & 7) << 28));
}

extern "C" int b200_valuenet_forward(b200_engine *e, const int8_t *states, int k, float *v, float *var) {
    if (!e || !states || !v || !var || k < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (k >= (1 << 28)) return fail(B200_ERR_BAD_ARG, "k too large");
    CK(cudaSetDevice(e->cfg.device));
    uint32_t *d_keys = nullptr; uint2 *d_req = nullptr; int32_t *d_n = nullptr; float2 *d_out = nullptr;
    size_t kp = ((size_t)k + 7) & ~(size_t)7;
    Scratch tmp;
    if (int rc = stage_boards(e, tmp, states, k, kp, &d_keys, &d_req, &d_n)) return rc;
    CK(tmp.get(&d_out, kp * 8));
    // keys are addressed as keys[(game * M + obs)]: with game = i/8 we pass M = 0 so that only obs (= i) indexes
    int rc = launch_net(e, d_req, d_n, d_keys, 0, d_out, kp);
    if (rc == B200_OK) {
        std::vector<float2> h(k);
        cudaError_t ce = cudaMemcpyAsync(h.data(), d_out, (size_t)k * 8, cudaMemcpyDeviceToHost, e->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
        if (ce != cudaSuccess) rc = fail(B200_ERR_CUDA, cudaGetErrorString(ce));
        else for (int i = 0; i < k; ++i) { v[i] = h[i].x; var[i] = h[i].y; }
    }
    cudaStreamSynchronize(e->stream);
    return rc;
}

// development / test aid: the conv stack's output (flatten input of fc1) in torch order c*56 + y*4 + x, for either path
extern "C" int b200_debug_act3(b200_engine *e, const int8_t *states, int k, float *out) {
    if (!e || !states || !out || k < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    std::vector<float> v(k), var(k);
    int rc = b200_valuenet_forward(e, states, k, v.data(), var.data());   // leaves act3 of these k boards in the scratch buffers
    if (rc) return rc;
    if (e->cfg.eval_kind == B200_EVAL_NET_TC) {
        std::vector<uint8_t> h(e->act3_tiles * TcfPipe::ACT_TILE_BYTES);
        CK(cudaMemcpy(h.data(), e->d_act3_tc, h.size(), cudaMemcpyDeviceToHost));
        for (int r = 0; r < k; ++r)
            for (int kp = 0; kp < 1792; ++kp) {
                int p = kp >> 5, c = kp & 31;
                float sum = 0.f;
                for (int s = 1; s >= 0; --s) {
                    size_t off = ((((size_t)s * e->act3_tiles + (r >> 7)) * ACT3_KCHUNKS + (kp >> 3)) * 128 + (r & 127)) * 16 + (kp & 7) * 2;
                    uint16_t hb; memcpy(&hb, &h[off], 2);
                    sum += host_half_f(hb);
                }
                out[(size_t)r * 1792 + c * 56 + p] = sum / TC_SCALE_A;
            }
        return B200_OK;
    }
    std::vector<float> h((size_t)k * 1792);
    CK(cudaMemcpy(h.data(), e->d_act3, h.size() * 4, cudaMemcpyDeviceToHost));
    for (int r = 0; r < k; ++r)
        for (int y = 0; y < 14; ++y)
            for (int c = 0; c < 32; ++c)
                for (int x = 0; x < 4; ++x) out[(size_t)r * 1792 + c * 56 + y * 4 + x] = h[(size_t)r * 1792 + (y * 32 + c) * 4 + x];
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- standalone env
static int env_stream_op(uint32_t *recs, const int32_t *actions, int8_t *state_out, int n) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    uint32_t *d = nullptr; int32_t *da = nullptr; int8_t *ds = nullptr;
    Scratch tmp;
    CK(tmp.get(&d, (size_t)n * REC_WORDS * 4));
    CK(cudaMemcpy(d, recs, (size_t)n * REC_WORDS * 4, cudaMemcpyHostToDevice));
    if (actions) {
        CK(tmp.get(&da, (size_t)n * 4));
        CK(cudaMemcpy(da, actions, (size_t)n * 4, cudaMemcpyHostToDevice));
        k_env_step<<<(n + 127) / 128, 128>>>(d, da, n);
        CK(cudaGetLastError());
        CK(cudaMemcpy(recs, d, (size_t)n * REC_WORDS * 4, cudaMemcpyDeviceToHost));
    }
    if (state_out) {
        CK(tmp.get(&ds, (size_t)n * 200));
        k_env_state<<<(n + 127) / 128, 128>>>(d, ds, n);
        CK(cudaGetLastError());
        CK(cudaMemcpy(state_out, ds, (size_t)n * 200, cudaMemcpyDeviceToHost));
    }
    return B200_OK;
}

extern "C" int b200_tetris_new(uint32_t *recs, int n, int app, int scoring, int randomizer, const uint32_t *seeds, int reset) {
    if (!recs || n < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    uint32_t *d = nullptr, *ds = nullptr;
    Scratch tmp;
    CK(tmp.get(&d, (size_t)n * REC_WORDS * 4));
    if (reset) CK(cudaMemcpy(d, recs, (size_t)n * REC_WORDS * 4, cudaMemcpyHostToDevice));
    if (seeds && !reset) { CK(tmp.get(&ds, (size_t)n * 4)); CK(cudaMemcpy(ds, seeds, (size_t)n * 4, cudaMemcpyHostToDevice)); }
    k_new_games<<<(n + 127) / 128, 128>>>(d, n, app, scoring, randomizer, ds, reset);
    CK(cudaGetLastError());
    CK(cudaMemcpy(recs, d, (size_t)n * REC_WORDS * 4, cudaMemcpyDeviceToHost));
    return B200_OK;
}

extern "C" int b200_tetris_step(uint32_t *recs, const int32_t *actions, int n) {
    if (!recs || !actions || n < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    return env_stream_op(recs, actions, nullptr, n);
}
extern "C" int b200_tetris_state(const uint32_t *recs, int8_t *out, int n) {
    if (!recs || !out || n < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    return env_stream_op(const_cast<uint32_t *>(recs), nullptr, out, n);
}

// ---------------------------------------------------------------------------------------------------- core twins
struct TwinBufs {
    int32_t *child = nullptr, *visit = nullptr, *n2o = nullptr, *trace = nullptr, *out = nullptr;
    float *value = nullptr, *variance = nullptr, *score = nullptr, *zt = nullptr;
    uint32_t *rng = nullptr;
    std::vector<void *> all;
    ~TwinBufs() { for (void *p : all) cudaFree(p); }
    template <typename T> int up(T **d, const T *h, size_t n) {
        if (cudaMalloc((void **)d, (n ? n : 1) * sizeof(T)) != cudaSuccess) return 1;
        all.push_back(*d);
        if (h && n) return cudaMemcpy(*d, h, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess;
        return cudaMemset(*d, 0, (n ? n : 1) * sizeof(T)) != cudaSuccess;
    }
};

static int twin_arena(TwinBufs &b, Arena &A) {
    memset(&A, 0, sizeof(A));
    std::vector<float> h(ZTABLE_N);
    const double l2 = log(2.0), l22 = log(22.0), l41 = log(41.0);
    for (int n = 0; n < ZTABLE_N; ++n) {
        double t = (double)n, alpha = 1 - 1 / t;
        h[n] = (float)(10 * log(1 - log(-log(alpha) / l2) / l22) / l41);
    }
    if (b.up(&b.zt, h.data(), (size_t)ZTABLE_N)) return 1;
    A.ztable = b.zt;
    return 0;
}

#define TW(x) do { if (x) return fail(B200_ERR_CUDA, "twin: device allocation/copy failed"); } while (0)

extern "C" int b200_select_trace_obs(int index, const int32_t *child, const int32_t *visit, const float *value,
                                     const float *variance, const float *score, const int32_t *n_to_o, int M, int low,
                                     uint32_t *rng_state, int32_t *trace_out, int max_trace, int32_t *trace_len) {
    if (!child || !visit || !value || !variance || !score || !n_to_o || !trace_out || !trace_len || index < 0 || index >= M)
        return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; Arena A;
    TW(twin_arena(b, A));
    uint32_t seed = rng_state ? *rng_state : 0x2545F491u;
    TW(b.up(&b.child, child, (size_t)M * 7)); TW(b.up(&b.visit, visit, (size_t)M)); TW(b.up(&b.value, value, (size_t)M));
    TW(b.up(&b.variance, variance, (size_t)M)); TW(b.up(&b.score, score, (size_t)M)); TW(b.up(&b.n2o, n_to_o, (size_t)M));
    TW(b.up(&b.trace, (const int32_t *)nullptr, (size_t)max_trace)); TW(b.up(&b.out, (const int32_t *)nullptr, 16)); TW(b.up(&b.rng, &seed, 1));
    TwinArgs t{b.child, b.visit, b.value, b.variance, b.score, b.n2o, b.trace, b.rng, b.out};
    k_twin_select<<<1, 32>>>(A, t, index, low, max_trace);
    CK(cudaGetLastError());
    int32_t out[2];
    CK(cudaMemcpy(out, b.out, 8, cudaMemcpyDeviceToHost));
    if (out[1] != ST_OK) return fail(B200_ERR_TRACE_FULL, "trace longer than max_trace");
    CK(cudaMemcpy(trace_out, b.trace, (size_t)out[0] * 4, cudaMemcpyDeviceToHost));
    if (rng_state) CK(cudaMemcpy(rng_state, b.rng, 4, cudaMemcpyDeviceToHost));
    *trace_len = out[0];
    return B200_OK;
}

extern "C" int b200_get_unique_child_obs(int index, const int32_t *child, const float *score, const int32_t *n_to_o, int M,
                                         int32_t *c_nodes, int32_t *c_obs, int32_t *k_out) {
    if (!child || !score || !n_to_o || !c_nodes || !c_obs || !k_out || index < 0 || index >= M) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; Arena A;
    TW(twin_arena(b, A));
    TW(b.up(&b.child, child, (size_t)M * 7)); TW(b.up(&b.score, score, (size_t)M)); TW(b.up(&b.n2o, n_to_o, (size_t)M));
    TW(b.up(&b.out, (const int32_t *)nullptr, 16));
    TwinArgs t{b.child, nullptr, nullptr, nullptr, b.score, b.n2o, nullptr, nullptr, b.out};
    k_twin_unique<<<1, 32>>>(A, t, index);
    CK(cudaGetLastError());
    int32_t out[16];
    CK(cudaMemcpy(out, b.out, 64, cudaMemcpyDeviceToHost));
    *k_out = out[0];
    for (int i = 0; i < out[0]; ++i) { c_nodes[i] = out[1 + i]; c_obs[i] = out[8 + i]; }
    return B200_OK;
}

static int twin_backup_common(TwinBufs &b, const int32_t *trace, int D, int32_t *visit, float *value, float *variance,
                              const int32_t *n_to_o, const float *score, int M) {
    if (b.up(&b.trace, trace, (size_t)D) || b.up(&b.visit, (const int32_t *)visit, (size_t)M) || b.up(&b.value, (const float *)value, (size_t)M) ||
        b.up(&b.variance, (const float *)variance, (size_t)M) || b.up(&b.n2o, n_to_o, (size_t)M) || b.up(&b.score, score, (size_t)M)) return 1;
    return 0;
}
static int twin_backup_fetch(TwinBufs &b, int32_t *visit, float *value, float *variance, int M) {
    if (cudaMemcpy(visit, b.visit, (size_t)M * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    if (cudaMemcpy(value, b.value, (size_t)M * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    if (cudaMemcpy(variance, b.variance, (size_t)M * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    return 0;
}

extern "C" int b200_backup_trace_obs(const int32_t *trace, int D, int32_t *visit, float *value, float *variance,
                                     const int32_t *n_to_o, const float *score, int M, double v, double var, double gamma) {
    if (!trace || D < 1 || !visit || !value || !variance || !n_to_o || !score) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; Arena A;
    TW(twin_arena(b, A));
    TW(twin_backup_common(b, trace, D, visit, value, variance, n_to_o, score, M));
    TwinArgs t{nullptr, b.visit, b.value, b.variance, b.score, b.n2o, b.trace, nullptr, nullptr};
    k_twin_backup<<<1, 1>>>(A, t, D, v, var, gamma, 0);
    CK(cudaGetLastError());
    TW(twin_backup_fetch(b, visit, value, variance, M));
    return B200_OK;
}

extern "C" int b200_backup_trace_obs_LP(const int32_t *trace, int D, int32_t *visit, float *value, float *variance,
                                        const int32_t *n_to_o, const float *score, const uint8_t *end, int M,
                                        const int32_t *c_nodes, const int32_t *c_obs, int k, const float *v, const float *var,
                                        double gamma, int mixture, int averaged) {
    if (!trace || D < 1 || !visit || !value || !variance || !n_to_o || !score || !end || k < 0 || k > 7) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; Arena A;
    TW(twin_arena(b, A));
    TW(twin_backup_common(b, trace, D, visit, value, variance, n_to_o, score, M));
    uint8_t *d_end = nullptr; int32_t *d_cn = nullptr, *d_co = nullptr; float *d_v = nullptr, *d_var = nullptr;
    TW(b.up(&d_end, end, (size_t)M)); TW(b.up(&d_cn, c_nodes, (size_t)k)); TW(b.up(&d_co, c_obs, (size_t)k));
    TW(b.up(&d_v, v, (size_t)k)); TW(b.up(&d_var, var, (size_t)k));
    TwinArgs t{nullptr, b.visit, b.value, b.variance, b.score, b.n2o, b.trace, nullptr, nullptr};
    k_twin_backup_lp<<<1, 1>>>(A, t, D, d_end, d_cn, d_co, k, d_v, d_var, gamma, mixture, averaged);
    CK(cudaGetLastError());
    TW(twin_backup_fetch(b, visit, value, variance, M));
    return B200_OK;
}

extern "C" int b200_get_all_childs(int index, const int32_t *child, int M, uint8_t *mark) {
    if (!child || !mark || index < 0 || index >= M) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b;
    uint8_t *d_mark = nullptr; int32_t *d_q = nullptr;
    TW(b.up(&b.child, child, (size_t)M * 7)); TW(b.up(&d_mark, (const uint8_t *)nullptr, (size_t)M)); TW(b.up(&d_q, (const int32_t *)nullptr, (size_t)M));
    k_twin_all_childs<<<1, 32>>>(b.child, M, index, d_mark, d_q);
    CK(cudaGetLastError());
    CK(cudaMemcpy(mark, d_mark, (size_t)M, cudaMemcpyDeviceToHost));
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- distributional cores (a16)
extern "C" int b200_dist_shift_distribution(const float *dist, int bins, double x, double vmin, double vmax, float *out) {
    if (!dist || !out || bins < 1 || bins > 4096) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; float *d_in = nullptr, *d_out = nullptr;
    TW(b.up(&d_in, dist, (size_t)bins)); TW(b.up(&d_out, (const float *)nullptr, (size_t)bins));
    k_dist_shift<<<1, 1>>>(d_in, bins, x, vmin, vmax, d_out);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, d_out, (size_t)bins * 4, cudaMemcpyDeviceToHost));
    return B200_OK;
}

extern "C" int b200_dist_mean_variance(const float *dist, int bins, double vmin, double vmax, double *mean, double *var) {
    if (!dist || !mean || !var || bins < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; float *d_in = nullptr; double *d_out = nullptr;
    TW(b.up(&d_in, dist, (size_t)bins)); TW(b.up(&d_out, (const double *)nullptr, 2));
    k_dist_mean_variance<<<1, 1>>>(d_in, bins, vmin, vmax, d_out);
    CK(cudaGetLastError());
    double h[2];
    CK(cudaMemcpy(h, d_out, 16, cudaMemcpyDeviceToHost));
    *mean = h[0]; *var = h[1];
    return B200_OK;
}

extern "C" int b200_dist_select_trace(int index, const int32_t *child, const float *node_stats, int M, int low, uint32_t *rng_state,
                                      int32_t *trace_out, int max_trace, int32_t *trace_len) {
    if (!child || !node_stats || !trace_out || !trace_len || index < 0 || index >= M) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; float *d_ns = nullptr; int32_t *d_len = nullptr;
    uint32_t seed = rng_state ? *rng_state : 0x2545F491u;
    TW(b.up(&b.child, child, (size_t)M * 7)); TW(b.up(&d_ns, node_stats, (size_t)M * 5)); TW(b.up(&b.trace, (const int32_t *)nullptr, (size_t)max_trace));
    TW(b.up(&b.rng, &seed, 1)); TW(b.up(&d_len, (const int32_t *)nullptr, 1));
    k_dist_select<<<1, 1>>>(index, b.child, d_ns, low, b.trace, max_trace, b.rng, d_len);
    CK(cudaGetLastError());
    int32_t n = 0;
    CK(cudaMemcpy(&n, d_len, 4, cudaMemcpyDeviceToHost));
    if (n < 0) return fail(B200_ERR_TRACE_FULL, "trace longer than max_trace");
    CK(cudaMemcpy(trace_out, b.trace, (size_t)n * 4, cudaMemcpyDeviceToHost));
    if (rng_state) CK(cudaMemcpy(rng_state, b.rng, 4, cudaMemcpyDeviceToHost));
    *trace_len = n;
    return B200_OK;
}

extern "C" int b200_dist_backup_trace(const int32_t *trace, int D, float *node_stats, float *node_dist, int M, int bins, double r,
                                      const float *dist, double vmin, double vmax) {
    if (!trace || D < 1 || !node_stats || !node_dist || !dist || bins < 1) return fail(B200_ERR_BAD_ARG, "bad argument");
    if (b200_device_count() == 0) return fail(B200_ERR_CUDA, "no CUDA device: this library has no CPU path");
    TwinBufs b; float *d_ns = nullptr, *d_nd = nullptr, *d_dist = nullptr, *d_scr = nullptr;
    TW(b.up(&b.trace, trace, (size_t)D)); TW(b.up(&d_ns, (const float *)node_stats, (size_t)M * 5)); TW(b.up(&d_nd, (const float *)node_dist, (size_t)M * bins));
    TW(b.up(&d_dist, dist, (size_t)bins)); TW(b.up(&d_scr, (const float *)nullptr, (size_t)bins));
    k_dist_backup<<<1, 1>>>(b.trace, D, d_ns, d_nd, bins, r, d_dist, vmin, vmax, d_scr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(node_stats, d_ns, (size_t)M * 5 * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(node_dist, d_nd, (size_t)M * bins * 4, cudaMemcpyDeviceToHost));
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- replay samples
__global__ void k_collect_samples(Arena A, int min_visits, uint8_t *out, int capacity, int32_t *count) {
    size_t n = (size_t)A.G * A.M;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        int4 st = A.stat[i];
        if (st.x < min_visits || st.w != 0 || st.x == 0) continue;      // ValueSim.py:143-144 (visit < min or end)
        int slot = atomicAdd(count, 1);
        if (slot >= capacity) continue;
        uint8_t *dst = out + (size_t)slot * 212;
        const uint32_t *k = A.key + i * KEY_WORDS;
        for (int r = 0; r < 20; ++r) {
            uint32_t row = (k[r >> 1] >> ((r & 1) * 16)) & 0x3ffu;
            for (int c = 0; c < 10; ++c) dst[r * 10 + c] = (uint8_t)((row >> c) & 1u);
        }
        for (int j = 0; j < 4; ++j) dst[(k[10] >> (8 * j)) & 0xffu] = 0xff;    // int8 -1
        float f[3] = {__int_as_float(st.y), __int_as_float(st.z), (float)st.x};
        memcpy(dst + 200, f, 12);
    }
}

// Online replay memory (agents/ValueSim.py:14-37, agent.cpp:588-617): allocate `capacity` rows; k_gc appends to it.
extern "C" int b200_replay_enable(b200_engine *e, int min_visits, int capacity) {
    if (!e || capacity < 1 || min_visits < 0) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    if (e->A.replay) return fail(B200_ERR_BAD_ARG, "replay memory already enabled");
    // twice the capacity is allocated: accumulation policy 0 (b200_replay_policy) stages the rows of a collection past memory_size before its
    // random drop decides which of them stay (agent.cpp:800-801); k_gc itself never stores past A.replay_cap
    if (dalloc(e, &e->A.replay, (size_t)2 * capacity * 212) || dalloc(e, &e->A.replay_count, 1)) return B200_ERR_CUDA;
    e->replay_alloc = 2 * capacity;
    e->A.replay_cap = capacity; e->A.replay_min_visits = min_visits;
    e->rp.memory_size = capacity;
    drop_step_graph(e);
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// Hand the stored rows to the trainer / the all-gather: copies min(count, capacity) rows to out_dev (DEVICE) and empties the memory
// (memory_index = 0 after training, ValueSim.py:183 / agent.cpp:700).
extern "C" int b200_replay_drain_dev(b200_engine *e, void *out_dev, int capacity, int32_t *count_out) {
    if (!e || !out_dev || !count_out || !e->A.replay) return fail(B200_ERR_BAD_ARG, "replay memory not enabled / bad argument");
    CK(cudaSetDevice(e->cfg.device));
    int32_t n = 0;
    CK(cudaMemcpyAsync(&n, e->A.replay_count, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (n > e->A.replay_cap) n = e->A.replay_cap;
    if (n > capacity) n = capacity;
    if (n > 0) CK(cudaMemcpyAsync(out_dev, e->A.replay, (size_t)n * 212, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaMemsetAsync(e->A.replay_count, 0, 4, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    *count_out = n;
    return B200_OK;
}

extern "C" int b200_collect_samples_dev(b200_engine *e, int min_visits, void *out_dev, int capacity, int32_t *count_out) {
    if (!e || !out_dev || capacity < 0 || !count_out) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    if (!e->d_sample_count) { if (dalloc(e, &e->d_sample_count, 1)) return B200_ERR_CUDA; }
    CK(cudaMemsetAsync(e->d_sample_count, 0, 4, e->stream));
    k_collect_samples<<<e->n_sm * 4, 256, 0, e->stream>>>(e->A, min_visits, (uint8_t *)out_dev, capacity, e->d_sample_count);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(count_out, e->d_sample_count, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (*count_out > capacity) *count_out = capacity;
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------- replay-memory policies (SURVEY 8f.1)
static int rp_count(b200_engine *e, int32_t *n) {
    CK(cudaMemcpyAsync(n, e->A.replay_count, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (*n > e->A.replay_cap) *n = e->A.replay_cap;
    return B200_OK;
}
static int rp_set_count(b200_engine *e, int32_t n) {
    CK(cudaMemcpyAsync(e->A.replay_count, &n, 4, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}
static int rp_scratch(b200_engine *e) {
    if (e->d_rp_tmp) return B200_OK;
    if (dalloc(e, &e->d_rp_tmp, (size_t)e->replay_alloc * 212, false) || dalloc(e, &e->d_rp_keep, (size_t)e->replay_alloc, false) ||
        dalloc(e, &e->d_rp_vis, (size_t)e->replay_alloc, false) || dalloc(e, &e->d_rp_kept, 1)) return B200_ERR_CUDA;
    return B200_OK;
}
// rows [lo, hi) with keep[i] != 0 are packed, in order, at lo, lo+1, ...; everything else in the memory stays as it is (the reference compacts
// in place by copying downwards, so positions past the packed rows keep their old content).  Returns the number of packed rows.
static int rp_compact(b200_engine *e, const std::vector<uint8_t> &keep, int lo, int hi, int *kept) {
    int rc = rp_scratch(e);
    if (rc) return rc;
    CK(cudaMemcpyAsync(e->d_rp_keep, keep.data(), (size_t)hi, cudaMemcpyHostToDevice, e->stream));
    k_replay_compact<<<1, 1024, 0, e->stream>>>(e->A.replay, e->d_rp_keep, lo, hi, e->d_rp_tmp, e->d_rp_kept);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(kept, e->d_rp_kept, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (*kept > 0) CK(cudaMemcpyAsync(e->A.replay + (size_t)lo * 212, e->d_rp_tmp + (size_t)lo * 212, (size_t)*kept * 212, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// OnlineMCTSAgent(accumulation_policy, episodes_per_train, memory_growth_rate) agent.cpp:588-617; memory_size / min_visit = b200_replay_enable's
extern "C" int b200_replay_policy(b200_engine *e, int policy, int episodes_per_train, int memory_growth_rate) {
    if (!e || !e->A.replay || policy < 0 || policy > 3 || episodes_per_train < 1 || memory_growth_rate < 0) return fail(B200_ERR_BAD_ARG, "replay memory not enabled / bad policy");
    CK(cudaSetDevice(e->cfg.device));
    ReplayPolicy fresh;
    fresh.policy = policy; fresh.memory_size = e->rp.memory_size; fresh.episodes_per_train = episodes_per_train; fresh.memory_growth_rate = memory_growth_rate;
    e->rp = fresh;
    e->A.replay_cap = policy == 0 ? e->replay_alloc : e->rp.memory_size;      // policy 0: rows are staged past memory_size until the drop has decided
    drop_step_graph(e);
    return rp_set_count(e, 0);
}

// weighted_trimming(percentile) agent.cpp:710-749 (literally, including that the first removed row is not subtracted from memory_index)
static int rp_weighted_trimming(b200_engine *e, double percentile) {
    ReplayPolicy &P = e->rp;
    const int N = P.memory_size;
    int rc = rp_scratch(e);
    if (rc) return rc;
    k_replay_visits<<<(N + 255) / 256, 256, 0, e->stream>>>(e->A.replay, N, e->d_rp_vis);
    std::vector<float> vis(N);
    CK(cudaMemcpyAsync(vis.data(), e->d_rp_vis, (size_t)N * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    std::vector<int> weights(N);
    for (int i = 0; i < N; ++i) weights[i] = (int)vis[i];
    std::sort(weights.begin(), weights.end());
    const int threshold = weights[(int)(N * percentile)];
    int idx_fill = -1;
    for (int i = 0; i < N; ++i) if (vis[i] <= (float)threshold) { idx_fill = i; break; }
    std::vector<uint8_t> keep(N, 1);
    for (int i = idx_fill; i < N; ++i) if (vis[i] <= (float)threshold) keep[i] = 0;
    for (int i = idx_fill + 1; i < N; ++i) if (vis[i] <= (float)threshold) --P.memory_index;
    int kept = 0;
    return rp_compact(e, keep, idx_fill, N, &kept);
}

// random_trimming(fraction) agent.cpp:751-775: IntSampler(memory_size).sample(n) = std::shuffle of the persistent index vector, first n, sorted
static int rp_random_trimming(b200_engine *e, double fraction) {
    ReplayPolicy &P = e->rp;
    const int N = P.memory_size;
    if (P.sampler.empty()) { P.sampler.resize(N); std::iota(P.sampler.begin(), P.sampler.end(), 0); }
    std::shuffle(P.sampler.begin(), P.sampler.end(), P.mt);
    std::vector<int> indices(P.sampler.begin(), P.sampler.begin() + (int)(N * fraction));
    if (indices.empty()) return B200_OK;                          // (the reference reads indices.front() of an empty vector here: UB)
    std::sort(indices.begin(), indices.end());
    std::vector<uint8_t> keep(N, 1);
    for (int i : indices) keep[i] = 0;
    P.memory_index -= (int)indices.size();
    int kept = 0;
    return rp_compact(e, keep, indices.front(), N, &kept);
}

// The policy half of OnlineMCTSAgent::remove_nodes (agent.cpp:632-702), to be called after the collection(s) that stored rows — the reference
// runs it inside every remove_nodes(); a single-game engine calls it after every simulation step / update_root in which counter 3 (collections)
// moved and then reproduces the reference exactly; a batched run calls it once per move.  current_episode = Agent::current_episode
// (agent.cpp:69,279-280: games finished so far).  *train_now = the reference would call train(m_state, m_value, m_variance, m_visit, memory_index)
// now: drain the first *memory_index rows (b200_replay_peek_dev), train, then b200_replay_policy_trained().
extern "C" int b200_replay_policy_step(b200_engine *e, int64_t current_episode, int32_t *train_now, int32_t *memory_index) {
    if (!e || !train_now || !memory_index || e->rp.policy < 0) return fail(B200_ERR_BAD_ARG, "no replay policy configured");
    CK(cudaSetDevice(e->cfg.device));
    ReplayPolicy &P = e->rp;
    int32_t count = 0;
    int rc = rp_count(e, &count);
    if (rc) return rc;
    const int cur = (int)current_episode;
    if (P.policy == 0) {
        // store_nodes' drop (agent.cpp:798-801), applied to the rows this collection staged, in their order: ++accumulated_nodes; a row is dropped
        // with probability memory_drop_prob; storing stops when the memory is full (:817)
        std::vector<uint8_t> keep((size_t)std::max(count, 1), 1);
        int kept_total = P.memory_index;
        bool full = kept_total >= P.memory_size;
        for (int i = P.memory_index; i < count; ++i) {
            if (full) { keep[i] = 0; continue; }
            ++P.accumulated_nodes;
            if (P.unif(P.mt) < P.memory_drop_prob) { keep[i] = 0; continue; }
            if (++kept_total == P.memory_size) full = true;
        }
        if (count > P.memory_index) {
            int kept = 0;
            rc = rp_compact(e, keep, P.memory_index, count, &kept);
            if (rc) return rc;
        }
        P.memory_index = kept_total;
        rc = rp_set_count(e, P.memory_index);
        if (rc) return rc;
    } else {
        P.memory_index = count < P.memory_size ? count : P.memory_size;
    }
    bool pass = false;
    const int diff = cur - P.last_training_episode;
    if (P.policy == 0) {
        if (P.last_accumulation_episode != cur) {
            P.nodes_per_episode.push_back(P.accumulated_nodes);
            if ((int)P.nodes_per_episode.size() > P.episodes_per_train) P.nodes_per_episode.pop_front();
            const int sum = std::accumulate(P.nodes_per_episode.begin(), P.nodes_per_episode.end(), 0);
            P.memory_drop_prob = std::max(0., 1. - double(P.memory_size) / sum);
            P.accumulated_nodes = 0;
            P.last_accumulation_episode = cur;
        }
        pass = diff >= P.episodes_per_train;
        if (!pass && P.memory_index >= P.memory_size) { rc = rp_random_trimming(e, 0.01); if (rc) return rc; rc = rp_set_count(e, P.memory_index); if (rc) return rc; }
    } else if (P.policy == 1) {
        pass = diff >= P.episodes_per_train;
        if (!pass && P.memory_index >= P.memory_size) { rc = rp_weighted_trimming(e, 0.01); if (rc) return rc; rc = rp_set_count(e, P.memory_index); if (rc) return rc; }
    } else if (P.policy == 2) {
        pass = diff >= P.episodes_per_train || P.memory_index >= P.memory_size;
    } else {
        const int m_size = std::min(P.n_trains * P.memory_growth_rate, P.memory_size);
        pass = P.memory_index >= m_size;
    }
    *train_now = pass ? 1 : 0;
    *memory_index = P.memory_index;
    return B200_OK;
}

// after train(...): ++n_trains; memory_index = 0; last_training_episode = current_episode (agent.cpp:697-701)
extern "C" int b200_replay_policy_trained(b200_engine *e, int64_t current_episode) {
    if (!e || e->rp.policy < 0) return fail(B200_ERR_BAD_ARG, "no replay policy configured");
    CK(cudaSetDevice(e->cfg.device));
    e->rp.n_trains += 1;
    e->rp.memory_index = 0;
    e->rp.last_training_episode = (int)current_episode;
    return rp_set_count(e, 0);
}

// Append n rows (HOST, 212 bytes each, the format k_gc stores) to the memory exactly as a collection would: in order, until the memory is full
// (agent.cpp:817).  Seeds the memory from a dump file (ValueSim.py:176-177) or from another process; the policy tests script collections with it.
extern "C" int b200_replay_append(b200_engine *e, const uint8_t *rows, int n) {
    if (!e || !e->A.replay || (n > 0 && !rows) || n < 0) return fail(B200_ERR_BAD_ARG, "replay memory not enabled / bad argument");
    CK(cudaSetDevice(e->cfg.device));
    int32_t count = 0;
    int rc = rp_count(e, &count);
    if (rc) return rc;
    int take = e->A.replay_cap - count;
    if (take > n) take = n;
    if (take > 0) CK(cudaMemcpyAsync(e->A.replay + (size_t)count * 212, rows, (size_t)take * 212, cudaMemcpyHostToDevice, e->stream));
    return rp_set_count(e, count + (take > 0 ? take : 0));
}

// the first n rows of the memory, copied to a DEVICE buffer without emptying it (the arrays the reference hands to train(): m_state ... [:memory_index])
extern "C" int b200_replay_peek_dev(b200_engine *e, void *out_dev, int n) {
    if (!e || !out_dev || n < 0 || !e->A.replay || n > e->replay_alloc) return fail(B200_ERR_BAD_ARG, "bad argument");
    CK(cudaSetDevice(e->cfg.device));
    if (n > 0) CK(cudaMemcpyAsync(out_dev, e->A.replay, (size_t)n * 212, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}
