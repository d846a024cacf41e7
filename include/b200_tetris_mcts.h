/*
 * b200_tetris_mcts.h — C-ABI of the B200-native batched Tetris-MCTS engine (libb200_tetris_mcts.so).
 *
 * This is the drop-in boundary for the reference's per-move simulation loop.  Every entry point names the
 * reference interface it replaces (file:line in hrpan/tetris_mcts @ 7f24f8d).  Conventions:
 *   - extern "C", plain pointers and sizes, no C++/torch types; the caller owns every buffer it passes;
 *   - pointers are HOST pointers unless the name says `_dev`;
 *   - every function returns 0 on success or a B200_ERR_* code; b200_last_error() gives the text;
 *   - one host thread per engine; all work of an engine is issued on ONE CUDA stream: its own, or the caller's (b200_engine_set_stream);
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns B200_ERR_CUDA.
 * Games travel as the 80-byte packed record of SPEC_PYTETRIS.md §6 (20 uint32 words).
 */
#ifndef B200_TETRIS_MCTS_H
#define B200_TETRIS_MCTS_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_BAD_ARG 1
#define B200_ERR_CUDA 2
#define B200_ERR_ARENA_FULL 3   /* reference: "MAX_NODES EXCEEDED" then UB, agents/cppmodule/agent.cpp:227-231 */
#define B200_ERR_TRACE_FULL 4
#define B200_ERR_NO_WEIGHTS 5

#define B200_REC_WORDS 20
#define B200_KEY_WORDS 12
#define B200_N_ACTIONS 7        /* agents/cppmodule/core.h:17 */
#define B200_N_WEIGHTS 478342   /* model/model_vv.py:13-46 Net: state_dict order, PyTorch layouts, + out_ubound, out_lbound */

enum { B200_MODE_LP = 0,        /* agents/ValueSimLP.py:13-70 */
       B200_MODE_SINGLE = 1,    /* agents/ValueSim.py:52-94 */
       B200_MODE_VANILLA = 2,   /* agents/Vanilla.py:17-64 */
       B200_MODE_DIST = 3 };    /* agents/core_distributional.py:82-124 driven as agents/DistValueSimOnline.py:36-75 sketches */
enum { B200_EVAL_SYNTHETIC = 0, /* test evaluator (hash of the observation), shared with the CPU oracle */
       B200_EVAL_NET = 1,       /* model/model_vv.py Model_VV.inference, fp32 CUDA cores */
       B200_EVAL_NET_TC = 2 };  /* same network on tcgen05 tensor cores (fp16 x 2 operand split, 3 products per product); in B200_MODE_DIST:
                                   model/model_distributional.py on tcgen05 (csrc/distnet_tc.cuh) instead of the fp32 CUDA-core kernels */

typedef struct b200_engine b200_engine;

typedef struct {
    int32_t n_games;            /* concurrent, independent game trees */
    int32_t max_nodes;          /* per-game arena, agents/agent.py:36 / agents/ValueSim.py:16 */
    int32_t mode;               /* B200_MODE_* */
    int32_t low;                /* check_low threshold: 1 (ValueSimLP.py:27), 5 (Vanilla.py:27) */
    int32_t lp_end_from_obs;    /* 0: ValueSimLP.py:25 behaviour; 1: agent.cpp:538 */
    int32_t lp_var_gamma2;      /* 1: core.h:365; 0: agent.cpp:558 */
    int32_t stale_pop;          /* 1: reproduce agents/agent.py:229-232 literally */
    int32_t overflow_reset;     /* 0: arena full after GC is an error (reference: IndexError agent.py:99 / UB agent.cpp:227-231);
                                   1: drop that game's tree and re-root it at the live game (counter 7 counts these) */
    int32_t eval_kind;          /* B200_EVAL_* */
    int32_t trace_max;          /* longest root-to-leaf path stored (0 -> 512) */
    int32_t actions_per_drop, scoring, randomizer;   /* play.py:75 env_args */
    int32_t device;             /* CUDA device ordinal */
    uint32_t seed;              /* search RNG stream base (replaces libc rand(), core.h:62,76, and random.randint, Vanilla.py:52) */
    double gamma;               /* ValueSim.py:14 0.999 / Vanilla.py:9 0.99 */
    double rollout_variance;    /* Vanilla.py:54 1e3 / VanillaC.py:8 1e5 */
    int32_t dist_bins;          /* B200_MODE_DIST: atoms, DistValueSimOnline.py:13 (50) */
    double dist_vmin, dist_vmax;   /* value range, DistValueSimOnline.py:13 (0, 5000) */
} b200_config;

const char *b200_last_error(void);
int b200_device_count(void);

/* --- engine lifetime: replaces TreeAgent.__init__/init_array (agents/agent.py:36-88), Agent.close (:303-307) */
int b200_engine_create(const b200_config *cfg, b200_engine **out);
int b200_engine_destroy(b200_engine *e);
/* --- SURVEY 8(b).5 "explicit cudaStream_t" (no reference counterpart: the reference is synchronous CPU code).  cuda_stream is a
 *     cudaStream_t passed as void* so that this header needs no CUDA include: from now on ALL work of the engine (kernels, the captured
 *     simulation step, async copies, the event timers) is issued on it; NULL = a private non-blocking stream again (the default).  The
 *     engine drains its previous stream inside the call; the caller owns its stream.  The legacy default stream cannot be captured into
 *     a CUDA graph: with it the step falls back to direct launches.  b200_engine_get_stream returns the stream in use, so that a caller
 *     that produces or consumes `_dev` buffers on its own stream can order against it (cudaStreamWaitEvent). */
int b200_engine_set_stream(b200_engine *e, void *cuda_stream);
int b200_engine_get_stream(b200_engine *e, void **cuda_stream_out);

/* --- Model.load (model/model.py:163-174): weights = the state_dict tensors concatenated (B200_N_WEIGHTS floats) */
int b200_load_weights(b200_engine *e, const float *weights);

/* --- TreeAgent.update_root (agents/agent.py:296-301) for all games: recs[n_games][20] */
int b200_set_games(b200_engine *e, const uint32_t *recs);
int b200_get_games(b200_engine *e, uint32_t *recs);
int b200_update_root(b200_engine *e, int auto_reset);

/* --- TreeAgent.remove_nodes (agents/agent.py:246-257; a public method, also reached from new_node :96-97 when the free list is
 * empty): collect every game that has fewer than min_free free node slots (INT_MAX: every game), as one batched launch.
 * b200_set_gc_headroom(n > 0) makes b200_update_root / b200_play_move do that after re-rooting (the driver calling remove_nodes() between
 * moves whenever len(agent.available) < n; b200_set_games only re-roots); 0 (default) = only the reference's own call site, inside new_node. */
int b200_remove_nodes(b200_engine *e, int min_free);
int b200_set_gc_headroom(b200_engine *e, int min_free);

/* --- memory traffic only (no reference counterpart, no effect on any result): the PATH CACHE.  Consecutive simulations of a game walk almost
 * the same root-to-leaf path (select_trace_obs, core.h:167-224, restarts at the root every time); with the cache on, a walk leaves next to its
 * trace the row fields and the children's statistics of every level, the backup (core.h:226-381) refreshes the copies it changes and drops
 * the ones a transposition made stale, and the next walk serves every level that is still valid from one sequential line instead of two
 * dependent random accesses.  B200_MODE_LP with max_nodes <= 65536; 192 bytes x trace_max per game (entry 160 + own record 16 + child ids 16).  0 (default) = off. */
int b200_set_path_cache(b200_engine *e, int on);

/* --- TreeAgent.mcts (agents/ValueSimLP.py:13, ValueSim.py:52, Vanilla.py:17): `sims` simulations on every game */
int b200_run_sims(b200_engine *e, int sims);

/* --- TreeAgent.compute_stats / get_action (agents/agent.py:153-185): stats[n][3][7], action[n] */
int b200_get_stats(b200_engine *e, float *stats, int32_t *action);

/* --- Tetris.play on the engine's live games (play.py:150): actions[n]; NULL = the argmax actions of the last stats */
int b200_env_step(b200_engine *e, const int32_t *actions);

/* --- one whole move of play.py:118-177 for every game: mcts -> get_action -> play -> update_root (-> reset) */
int b200_play_move(b200_engine *e, int sims, int auto_reset, int32_t *actions_out, float *stats_out);

/* --- the episodes that ended inside b200_update_root(auto_reset) / b200_play_move since the last call (play.py:161-177 prints
 *     `Episode: .. Score: .. Lines Cleared: ..` from these numbers before game.reset()): out4[i] = {game, score, line_clears, episode};
 *     at most cap rows are copied, *count_out = episodes ended (the device log holds 4 * n_games rows between drains) */
int b200_finished_games(b200_engine *e, int32_t *out4, int cap, int32_t *count_out);

int b200_status(b200_engine *e, int32_t *status);            /* per-game 0 ok / B200_ERR_ARENA_FULL / B200_ERR_TRACE_FULL */
int b200_counters(b200_engine *e, uint64_t *out16);          /* 0 sims 1 expansions 2 eval requests 3 gcs 4 trace levels
                                                                5 rollout steps 6 new nodes 7 tree resets 8 games finished 9 score sum 10 lines sum
                                                                12 longest trace of the last b200_run_sims (not cumulative)
                                                                13 trace levels served by the path cache (of counter 4) */
int b200_sync(b200_engine *e);
int b200_timer_start(b200_engine *e);                        /* CUDA-event stopwatch on the engine's stream (sync, then record) */
int b200_timer_stop(b200_engine *e, float *ms);              /* record, wait, elapsed milliseconds since b200_timer_start */
int b200_set_timing(b200_engine *e, int on);                 /* CUDA-event timing of each phase on the engine's stream */
int b200_phase_ms(b200_engine *e, float *ms8, uint64_t *launches8);   /* 0 select+expand 1 conv 2 fc 3 backup 4 rollout 5 synth 6 stats/step/root 7 gc+resume */

/* --- the arena of one game in the reference's array layout (agents/agent.py:58-88); any pointer may be NULL */
int b200_export_game(b200_engine *e, int game, int32_t *child, float *score, int32_t *episode, int32_t *n2o,
                     int32_t *visit, float *value, float *variance, uint8_t *obs_end, uint32_t *game_recs,
                     uint32_t *obs_keys, int32_t *root, int32_t *last_trace, int32_t *last_trace_len);

/* --- Model_VV.inference (model/model_vv.py:210-217): states[k][200] int8 -> v[k], var[k] */
int b200_valuenet_forward(b200_engine *e, const int8_t *states, int k, float *v, float *var);

/* --- pyTetris.Tetris ctor / reset / play / getState for host-resident games (play.py:75-76,150,169,
 *     agents/agent.py:116).  b200_tetris_new: reset == 0 builds n fresh games (seeds[n] or NULL = default seed),
 *     reset != 0 applies Tetris.reset() to the n records in place (keeps each RNG stream, SPEC §4). */
int b200_tetris_new(uint32_t *recs, int n, int actions_per_drop, int scoring, int randomizer, const uint32_t *seeds, int reset);
int b200_tetris_step(uint32_t *recs, const int32_t *actions, int n);
int b200_tetris_state(const uint32_t *recs, int8_t *out, int n);

/* --- single-call twins of agents/cppmodule/core.cpp:20-26 on the reference's own arrays (mutated in place) */
int b200_select_trace_obs(int index, const int32_t *child, const int32_t *visit, const float *value,
                          const float *variance, const float *score, const int32_t *n_to_o, int M, int low,
                          uint32_t *rng_state, int32_t *trace_out, int max_trace, int32_t *trace_len);
int b200_backup_trace_obs(const int32_t *trace, int D, int32_t *visit, float *value, float *variance,
                          const int32_t *n_to_o, const float *score, int M, double v, double var, double gamma);
int b200_backup_trace_obs_LP(const int32_t *trace, int D, int32_t *visit, float *value, float *variance,
                             const int32_t *n_to_o, const float *score, const uint8_t *end, int M,
                             const int32_t *c_nodes, const int32_t *c_obs, int k, const float *v, const float *var,
                             double gamma, int mixture, int averaged);
int b200_get_unique_child_obs(int index, const int32_t *child, const float *score, const int32_t *n_to_o, int M,
                              int32_t *c_nodes, int32_t *c_obs, int32_t *k_out);
int b200_get_all_childs(int index, const int32_t *child, int M, uint8_t *mark);

/* --- distributional cores (agents/core_distributional.py, BASELINE config 5), operator level, reference array layout:
 *     node_stats f32[M][5] = {visit, mean, reward, variance, M2}, node_dist f32[M][bins], child int32[M][7] */
int b200_dist_shift_distribution(const float *dist, int bins, double x, double vmin, double vmax, float *out);     /* :12-36 */
int b200_dist_mean_variance(const float *dist, int bins, double vmin, double vmax, double *mean, double *var);     /* :48-63 */
int b200_dist_select_trace(int index, const int32_t *child, const float *node_stats, int M, int low, uint32_t *rng_state,
                           int32_t *trace_out, int max_trace, int32_t *trace_len);                                 /* :82-106 */
int b200_dist_backup_trace(const int32_t *trace, int D, float *node_stats, float *node_dist, int M, int bins, double r,
                           const float *dist, double vmin, double vmax);                                           /* :109-124 */

/* --- distributional engine (B200_MODE_DIST): Model.load / Model.inference of model/model_distributional.py:18-57 and the
 *     node-indexed arrays of one game.  weights: seq.conv1.w[32,1,4,4] b[32] seq.conv2.w[32,32,4,4] b[32] seq.fc1.w[128,2048]
 *     b[128] seq.fc_v.w[atoms,128] b[atoms] concatenated (the reference hard-codes a 22x10 input, model_distributional.py:27:
 *     the 20x10 observation gets two empty rows on top). */
int b200_load_dist_weights(b200_engine *e, const float *weights, int atoms);
int b200_distnet_forward(b200_engine *e, const int8_t *states, int k, int atoms, float *dist);
int b200_export_dist(b200_engine *e, int game, float *node_stats /* [M][5] */, float *node_dist /* [M][bins] */);

/* --- replay samples of the live search (ValueSim.store_nodes, agents/ValueSim.py:122-159): observations with
 *     visit >= min_visits and not end, packed as {int8 state[200], f32 value, f32 variance, f32 visit} = 212 B.
 *     out_dev is a DEVICE buffer of capacity*212 bytes (e.g. a torch tensor handed to the NCCL all-gather). */
int b200_collect_samples_dev(b200_engine *e, int min_visits, void *out_dev, int capacity, int32_t *count_out);

/* --- online replay memory (ValueSim.memory agents/ValueSim.py:14-37; OnlineMCTSAgent agent.cpp:588-617): when enabled, every
 *     garbage collection appends the observations it frees that have visit >= min_visits and are not `end`
 *     (store_nodes, ValueSim.py:122-159 / agent.cpp:777-819) until `capacity` rows are held.  b200_replay_drain_dev copies the
 *     rows to a DEVICE buffer (trainer input / NCCL all-gather block) and empties the memory (ValueSim.py:183). */
int b200_replay_enable(b200_engine *e, int min_visits, int capacity);
int b200_replay_drain_dev(b200_engine *e, void *out_dev, int capacity, int32_t *count_out);

/* --- the online agent's accumulation policies and memory trimming (OnlineMCTSAgent::remove_nodes agent.cpp:619-708: policies 0-3;
 *     weighted_trimming :710-749; random_trimming :751-775; store_nodes' random drop :800-801), on the memory b200_replay_enable created
 *     (memory_size = capacity, min_visit = min_visits).  b200_replay_policy_step = the decision the reference takes inside remove_nodes() after
 *     storing: call it after collections (single game: after every step / update_root in which counter 3 moved — then memory contents, trimming
 *     and the moments of training equal the compiled agent.cpp's; batched: once per move) with current_episode = games finished so far
 *     (agent.cpp:279-280).  *train_now != 0: train on the first *memory_index rows (b200_replay_peek_dev), then b200_replay_policy_trained. */
int b200_replay_policy(b200_engine *e, int accumulation_policy, int episodes_per_train, int memory_growth_rate);
int b200_replay_policy_step(b200_engine *e, int64_t current_episode, int32_t *train_now, int32_t *memory_index);
int b200_replay_policy_trained(b200_engine *e, int64_t current_episode);
int b200_replay_peek_dev(b200_engine *e, void *out_dev, int n_rows);
int b200_replay_append(b200_engine *e, const uint8_t *rows_host, int n_rows);   /* rows join the memory as a collection's would: in order, until it is full */

/* --- value-network training step (SURVEY 8f.2): Model_VV._loss / Model.train / Yogi.step / Model_VV.train_data of the reference
 *     (model/model_vv.py:94-153,227-231, model/model.py:52-119, model/yogi.py:39-90) on the device.  weights = the state_dict vector of
 *     b200_load_weights (PyTorch layouts); a batch is {states int8[n][200], value f32[n], variance f32[n], weight f32[n]} (the four arrays
 *     of ValueSim.memory, agents/ValueSim.py:25-30).  Host logic that stays on the host (validation split, batch sampling, early stopping,
 *     checkpoint files): tetris_mcts_b200/model/model_vv.py Model_VV.train_data. */
typedef struct b200_trainer b200_trainer;
const char *b200_trainer_last_error(void);
int b200_trainer_create(int device, const float *weights, int max_batch, b200_trainer **out);     /* Model_VV._init_model (model_vv.py:125-134) */
int b200_trainer_destroy(b200_trainer *t);
int b200_trainer_set_hyper(b200_trainer *t, double lr, double beta1, double beta2, double eps, double weight_decay);   /* Yogi(...) model_vv.py:132 */
int b200_trainer_set_out_ubound(b200_trainer *t, float ub_value, float ub_variance);             /* model_vv.py:227-231 */
int b200_trainer_get_weights(b200_trainer *t, float *weights_out);                               /* model.state_dict() */
int b200_trainer_set_weights(b200_trainer *t, const float *weights);                             /* model.load_state_dict() */
int b200_trainer_get_state(b200_trainer *t, float *exp_avg, float *exp_avg_sq, int64_t *step);   /* optimizer.state_dict(); step -1 = no state yet */
int b200_trainer_set_state(b200_trainer *t, const float *exp_avg, const float *exp_avg_sq, int64_t step);   /* load_state_dict; step < 0 = reset_optimizer */
int b200_trainer_get_grads(b200_trainer *t, float *grads_out);                                   /* p.grad of the last step, state_dict order (478338 floats) */
/* Model_VV._loss under no_grad on one chunk (Model.compute_loss, model/model.py:52-83): mean and population std of (weight *) logl; pred_out NULL or [n][2] */
int b200_trainer_loss(b200_trainer *t, const int8_t *states, const float *value, const float *variance, const float *weight, int n,
                      int weighted, double *loss, double *loss_std, float *pred_out);
/* Model.train (model/model.py:95-119): forward, loss, backward, gradient norm, clip when grad_clip > 0, Yogi step */
int b200_trainer_step(b200_trainer *t, const int8_t *states, const float *value, const float *variance, const float *weight, int n,
                      int weighted, double grad_clip, double *loss, double *loss_std, double *grad_norm);
/* the same step on a batch gathered ON THE DEVICE from 212-byte replay rows (b200_replay_drain_dev / the all-gather block): idx[n] (host) are row
 * indices (np.random.choice, model/model.py:207), weight = visit * weight_scale (weights / weights.mean(), model/model.py:186-187) */
int b200_trainer_step_rows_dev(b200_trainer *t, const void *rows_dev, int n_rows, const int32_t *idx, int n, float weight_scale,
                               int weighted, double grad_clip, double *loss, double *loss_std, double *grad_norm);

#ifdef __cplusplus
}
#endif
#endif
