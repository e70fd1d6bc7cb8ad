/*
 * lsm_b200.h - C ABI of the B200-native batched simulator for the per-step hot path of
 * Layered-Safe-MARL's `navigation_graph_safe` environment.
 *
 * Plain pointers and sizes only (no torch / ATen types). Every pointer inside lsm_buffers and
 * lsm_grid_desc is a DEVICE pointer; the caller (the Python B200GraphVecEnv, or any other host)
 * owns the memory. All launches go to the cudaStream_t passed as `stream` (void*; NULL = default).
 * No entry point synchronises the device.
 *
 * Every function returns 0 on success, a non-zero code otherwise, and then lsm_last_error()
 * describes the failure (thread-local string).
 *
 * What each entry point replaces in the reference (paths relative to the reference root):
 *   lsm_step     GraphSubprocVecEnv.step_async/step_wait  onpolicy/envs/env_wrappers.py:983-996
 *                + graphworker 'step' incl. auto-reset     onpolicy/envs/env_wrappers.py:851-875
 *                + MultiAgentGraphEnv.step                 multiagent/environment.py:963-1042
 *                + World.step / apply_safety_filter        multiagent/core.py:593-709
 *                + both safety handles                     multiagent/safety_filter.py:203-433
 *                + reward / goal / observation / graph     multiagent/custom_scenarios/navigation_graph_safe.py:576-994
 *   lsm_reset    GraphSubprocVecEnv.reset                  onpolicy/envs/env_wrappers.py:998-1005
 *                + MultiAgentGraphEnv.reset                multiagent/environment.py:1046-1074
 *                + reset_world / update_curriculum / random_scenario
 *                                                          navigation_graph_safe.py:264-366,1199-1367
 *   lsm_observe  the observation half of reset (used after lsm set_state style injection)
 *   lsm_set_value_grid / lsm_set_ttr_grid
 *                HjDataHandle.__init__                     multiagent/safety_filter.py:154-168
 *                TTR grid loading in make_world            navigation_graph_safe.py:128-138
 *   lsm_create   Scenario.make_world (constants only)      navigation_graph_safe.py:58-262
 *   lsm_safety_filter  both safety handles' apply_safety_filter for caller-owned states
 *                                                          multiagent/safety_filter.py:203-260, 378-433
 *   lsm_hj_lookup      get_value_of_relative_state + gradient  multiagent/safety_filter.py:192-201, 345-354
 *   lsm_edges_from_records  TransformerConvNet.process_adj on a learner minibatch of stored rollout rows, straight from
 *                      the stored emit records (no dense adjacency)  onpolicy/algorithms/utils/gnn.py:376-407
 */
#ifndef LSM_B200_H
#define LSM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSM_ABI_VERSION 5

enum { LSM_DYN_DOUBLE_INTEGRATOR = 0, LSM_DYN_AIRTAXI = 1 };

/* switches of multiagent/config.py:RewardBinaryConfig plus the make_world arguments that gate code */
enum {
    LSM_FLAG_SAFETY_VIOLATION = 1 << 0,
    LSM_FLAG_HJ_VALUE = 1 << 1,
    LSM_FLAG_POTENTIAL_CONFLICT = 1 << 2,
    LSM_FLAG_SEPARATION_DISTANCE_CURRICULUM = 1 << 3,
    LSM_FLAG_INITIAL_PHASE_USE_SAFETY_FILTER = 1 << 4,
    LSM_FLAG_DIFF_FROM_FILTERED_ACTION = 1 << 5,
    LSM_FLAG_USE_SAFETY_FILTER = 1 << 6,   /* the --use_safety_filter argument */
    LSM_FLAG_SHARED_REWARD = 1 << 7,       /* --collaborative */
    LSM_FLAG_USE_MASKING = 1 << 8,         /* --use_masking (required, reference quirk Q9) */
    LSM_FLAG_GRAPH_FEAT_GLOBAL = 1 << 9,   /* --graph_feat_type global: 7-wide observer-independent node features
                                              (navigation_graph_safe.py:1017-1036); default is 'relative' */
    LSM_FLAG_INTERP_FLOAT32 = 1 << 10      /* grid interpolation (hj_reachability Grid.interpolate: safety_filter.py:195,245,
                                              348,418, core.py:463, navigation_graph_safe.py:751) in float32 - position,
                                              weights and corner sum - as jax computes it without jax_enable_x64 (the
                                              reference never enables it); default: the same formula in float64.
                                              Both modes run the specialised pipeline on the shapes it is compiled for
                                              (float32 agent / pair kernels of their own) and the generic kernel on the
                                              others */
};

/* state layout: agent_f64[field][env][agent], agent_i32[field][env][agent],
 * landmarks[field][env][order*N + agent], env_f64[field][env], env_i32[field][env] */
enum {
    LSM_AF_X = 0, LSM_AF_Y, LSM_AF_S2 /* vx | theta */, LSM_AF_S3 /* vy | speed */,
    LSM_AF_P_DIST, LSM_AF_STATE_TIME, LSM_AF_MIN_REL_DIST, LSM_AF_GOAL_MIN_TIME,
    LSM_AF_TIMES_REQ_A, LSM_AF_TIMES_REQ_B, LSM_AF_DISTS_GOAL_A, LSM_AF_DISTS_GOAL_B,
    LSM_AF_DIST_LEFT, LSM_AF_EP_TRAVEL_DIST, LSM_AF_EP_MIN_DIST, LSM_AF_ACTION_DIFF,
    LSM_AF_COUNT
};
enum {
    LSM_AI_REACHED = 0, LSM_AI_DONE, LSM_AI_SAFETY_FILTERED, LSM_AI_DECONFLICT_IDX,
    LSM_AI_NUM_COLLISIONS, LSM_AI_EP_TRAVEL_LEN, LSM_AI_EP_CONFLICT, LSM_AI_EP_MULTI,
    LSM_AI_EP_DONE, LSM_AI_NUM_OBST_COLLISIONS /* world.num_obstacle_collisions (obstacle extension) */, LSM_AI_COUNT
};
enum { LSM_LF_X = 0, LSM_LF_Y, LSM_LF_HEADING, LSM_LF_SPEED, LSM_LF_SIN, LSM_LF_COS, LSM_LF_COUNT };
enum { LSM_EF_CURRICULUM_RATIO = 0, LSM_EF_COUNT };
enum { LSM_EI_CURRENT_STEP = 0, LSM_EI_RESET_COUNT, LSM_EI_PARITY, LSM_EI_JUST_RESET, LSM_EI_COUNT };
enum {
    LSM_EP_TRAVEL_TIME_MEAN = 0, LSM_EP_TRAVEL_DISTANCE_MEAN, LSM_EP_DONE_PERCENTAGE,
    LSM_EP_NUM_REACHED_GOAL_MEAN, LSM_EP_CONFLICT_PERCENTAGE, LSM_EP_MIN_DISTANCE_MEAN,
    LSM_EP_MIN_DISTANCE_MIN, LSM_EP_MULTIPLE_ENGAGEMENT_PERCENTAGE, LSM_EP_COUNT
};

/* terminal-step snapshot of the fields info_callback reads (navigation_graph_safe.py:386-450), written ONLY for an
 * environment that auto-resets in this step, before the reset overwrites its state: graphworker returns the terminal
 * step's infos and only appends the episode summary (onpolicy/envs/env_wrappers.py:861-874).
 * term_f64[field][env][agent], term_i32[field][env][agent], term_env_f64[env] = curriculum ratio of the finished episode */
enum {
    LSM_TF_X = 0, LSM_TF_Y, LSM_TF_MIN_REL_DIST, LSM_TF_DIST_LEFT, LSM_TF_TIMES_REQ_NEW, LSM_TF_TIMES_REQ_OLD,
    LSM_TF_DISTS_GOAL_NEW, LSM_TF_DISTS_GOAL_OLD, LSM_TF_GOAL_MIN_TIME, LSM_TF_COUNT
};
enum { LSM_TI_NUM_COLLISIONS = 0, LSM_TI_SAFETY_FILTERED, LSM_TI_NUM_OBST_COLLISIONS, LSM_TI_COUNT };

#define LSM_MAX_AGENTS 32
#define LSM_MAX_LANDMARKS 128
#define LSM_MAX_OBSTACLES 32
#define LSM_NUM_ACTIONS 25

typedef struct lsm_config {
    int32_t dynamics, num_agents, num_landmarks /* per agent */, episode_length;
    int32_t num_total_episode, num_internal_step;
    uint32_t flags;
    int32_t num_obstacles;        /* --num_obstacles. 0 in every shipped script; > 0 is a DECLARED EXTENSION (the reference raises,
                                     navigation_graph_safe.py:1064-1065,1087 / :975-989): obstacles are placed, collide and enter the
                                     distance matrix as the reference's own code does (:230-236,402-404,452-465,1204-1249,
                                     core.py:489-543); an obstacle is never disconnected and its 'relative' node features are the
                                     landmark builders' (utils.py:174-199,231-255) with heading 0, speed 0, entity type 2.
                                     Runs the generic fused kernel */
    double world_size;
    double dt, coordination_range, dist_thresh, heading_thresh, speed_thresh;
    double goal_speed_min, goal_speed_max, separation_distance_target;
    double engagement_distance_ref, engagement_ref_separation, cbf_rate, agent_max_speed;
    double goal_rew, safety_violation_rew, hj_value_rew, potential_conflict_rew;
    double diff_from_filtered_action_rew, min_reward, max_reward;
    double act_tab0[5], act_tab1[5];   /* np.linspace tables of environment.py:387-410 */
} lsm_config;

/* lsm_set_value_grid / lsm_set_ttr_grid refuse (code 2) a descriptor with a dimension of fewer than 2 nodes or with
 * 2^31 cells or more, before reading any array; a refused call leaves the grid bound before it in place. */
typedef struct lsm_grid_desc {
    int32_t ndim;
    int32_t shape[5];
    int32_t periodic[5];
    int32_t _pad;
    double lo[5], hi[5];
    double separation_distance;   /* separation distance the values encode */
    double ttr_max;
    const float *values;          /* DEVICE [prod(shape)], C order */
    const float *grads;           /* DEVICE [prod(shape)][ndim], or NULL */
} lsm_grid_desc;

typedef struct lsm_buffers {
    int64_t num_envs;
    int64_t env_id_base;          /* global index of env 0 of this shard (keys the reset RNG stream) */
    double *agent_f64;            /* [LSM_AF_COUNT][num_envs][N] */
    int32_t *agent_i32;           /* [LSM_AI_COUNT][num_envs][N] */
    double *landmarks;            /* [LSM_LF_COUNT][num_envs][N*L] */
    double *env_f64;              /* [LSM_EF_COUNT][num_envs] */
    int32_t *env_i32;             /* [LSM_EI_COUNT][num_envs] */
    /* outputs */
    float *obs;                   /* [num_envs][N][D]       D = 7 (DI) | 6 (airtaxi) */
    float *node_obs;              /* [num_envs][N][E][F]    F = 10 (DI) | 11 (airtaxi) | 7 (global features), E = N(1+L) + O */
    float *adj;                   /* [num_envs][N][E][E] */
    float *reward;                /* [num_envs][N] */
    uint8_t *done;                /* [num_envs][N] */
    double *safe_action;          /* [num_envs][N][2]  control applied in the last internal step */
    double *ep_info;              /* [num_envs][LSM_EP_COUNT]  summary written when an env resets */
    float *reward_individual;     /* [num_envs][N] or NULL: pre-sum reward when LSM_FLAG_SHARED_REWARD */
    /* terminal-step info snapshot of auto-resetting envs (all three NULL = not recorded) */
    double *term_f64;             /* [LSM_TF_COUNT][num_envs][N] */
    int32_t *term_i32;            /* [LSM_TI_COUNT][num_envs][N] */
    double *term_env_f64;         /* [num_envs] */
    double *obstacles;            /* [2][num_envs][O] obstacle x / y; required when num_obstacles > 0, ignored otherwise */
} lsm_buffers;

/* Launch-shape choices a caller may override (lsm_set_tuning, right after lsm_create; 0 / -1 = automatic). These are
 * the library's only knobs: it reads no environment variable. */
typedef struct lsm_tuning {
    int32_t chunks;               /* env ranges one step is split into on library-owned streams (1..16); 0 = automatic
                                     (4 from 0.4 GB of observations per step, else 1) */
    int32_t pair_placement;       /* where the next step's HJ pair values are computed: 0 behind the emit kernel,
                                     2 in front of the agent kernel, 3 between agent and emit kernel, 4 at the tail of the
                                     agent kernel itself (no pair kernel); -1 = automatic
                                     (0 for the 4-D grid, 3 for the 5-D grid) */
    int32_t packed_grid;          /* 1 corner-packed value table (one aligned chunk per lookup), 0 scattered gathers;
                                     -1 = automatic (packed when the table fits 2 GiB) */
    int32_t use_graph;            /* 1 replay a step's launches from a CUDA graph once the same parameter block repeats (one
                                     graph launch instead of 2-3 kernel launches: less host time per step and no host-side
                                     gap between the kernels of one step; ~1 us more device time per step on B200), 0 plain
                                     launches; -1 = automatic (plain launches). Single-range steps of the specialised
                                     pipeline only */
} lsm_tuning;

typedef struct lsm_launch_info {
    int32_t grid_blocks, block_threads, warps_per_block, envs_per_warp;
    int32_t smem_bytes_per_block, regs_per_thread, blocks_per_sm, sm_count;
    int32_t specialised;          /* 1: compile-time (dynamics, N, L) three-launch pipeline, 0: generic fused kernel */
    /* specialised pipeline only: the graph-emission kernel (one block per env) and the pair kernel */
    int32_t emit_block_threads, emit_smem_bytes_per_block, emit_regs_per_thread, emit_blocks_per_sm;
    int32_t pair_regs_per_thread;
    int32_t launches_per_step;    /* kernels one lsm_step launches in steady state */
    int32_t emit_record_bytes;    /* per-env record handed from the agent kernel to the emit kernel */
    int32_t chunks;               /* env ranges one lsm_step is split into (library-owned streams, fork/join by events); 1 = none */
    int32_t pair_placement;       /* next step's HJ pair values: 0 behind the emit kernel, 1 inside it, 2 in front of the agent kernel, 3 between the two; -1 none */
    int32_t graph_replays;        /* lsm_step calls served by a CUDA-graph launch so far (lsm_tuning.use_graph), saturating */
    int32_t graph_captures;       /* captures / in-place updates of that graph so far */
} lsm_launch_info;

typedef struct lsm_handle lsm_handle;

int lsm_abi_version(void);
const char *lsm_last_error(void);

int lsm_create(const lsm_config *cfg, lsm_handle **out);
int lsm_destroy(lsm_handle *h);
int lsm_set_value_grid(lsm_handle *h, const lsm_grid_desc *g);
int lsm_set_ttr_grid(lsm_handle *h, const lsm_grid_desc *g);
int lsm_set_tuning(lsm_handle *h, const lsm_tuning *t);
int lsm_bind_buffers(lsm_handle *h, const lsm_buffers *b);
int lsm_get_launch_info(lsm_handle *h, lsm_launch_info *out);

/* One env.step for every env (exactly one of action_idx / action_onehot non-NULL):
 *   action_idx    DEVICE int32 [num_envs][N] in [0,25)
 *   action_onehot DEVICE float [num_envs][N][25]; argmax (first maximum) is taken on device
 * episode is the `num_current_episode` the runner passes to envs.step; auto_reset != 0 reproduces
 * graphworker (reset an env whose agents are all done, keep the step's rewards/dones). */
int lsm_step(lsm_handle *h, const int32_t *action_idx, const float *action_onehot, int64_t episode,
             uint64_t seed, int auto_reset, void *stream);

/* env.reset(episode) for every env with env_mask[e] != 0 (DEVICE uint8, NULL = all). sample != 0
 * draws a new random scenario on device; sample == 0 keeps the injected agents / landmarks. The other envs keep their
 * state and outputs; with the fused edge output on (lsm_set_edge_output) their edges are written again, because the
 * offsets of every later graph move. */
int lsm_reset(lsm_handle *h, const uint8_t *env_mask, int64_t episode, uint64_t seed, int sample,
              void *stream);

/* Re-emit obs / node_obs / adj from the bound state without stepping. */
int lsm_observe(lsm_handle *h, void *stream);

/* Re-point the per-step OUTPUT arrays (any of them NULL = keep the current binding). Cheap (no allocation, no
 * launch): lets a device-resident rollout buffer receive every step directly in its slot for that step instead
 * of copying it there afterwards (the reference copies twice: np.stack in GraphSubprocVecEnv.step_wait,
 * env_wrappers.py:985-996, and .copy() in GraphReplayBuffer.insert, graph_buffer.py:223-228).
 * node_obs and adj must be 16-byte aligned. */
int lsm_set_output_buffers(lsm_handle *h, float *obs, float *node_obs, float *adj, float *reward, uint8_t *done);

/* Compact adjacency for HOST-facing callers (GraphSubprocVecEnv.step_wait returns host arrays,
 * onpolicy/envs/env_wrappers.py:983-996): the N observer matrices of one environment are ONE radius-thresholded E x E
 * distance matrix with observer-specific rows / columns zeroed (navigation_graph_safe.py:974-992). With both pointers
 * non-NULL the step kernels write, instead of the dense adj output,
 *   adj_base  DEVICE float    [num_envs][E][E]     thresholded distances, unmasked
 *   adj_keep  DEVICE uint32   [num_envs][N][W]     W = ceil(E / 32): bit e of observer i's words = entity e is connected
 * so that 1/N of the adjacency bytes cross PCIe; lsm_expand_adjacency_host rebuilds the dense array byte for byte.
 * Both NULL restores the dense output. Specialised (dynamics, N, L) configurations only, in either interpolation mode
 * (returns 6 otherwise). */
int lsm_set_compact_adjacency(lsm_handle *h, float *adj_base, uint32_t *adj_keep);

/* HOST function (no GPU work): adj[e][i][a][b] = keep_i[a] && keep_i[b] ? base[e][a][b] : 0 for e in [0, num_envs),
 * written by `threads` worker threads (<= 0: one per online core, at most 16) of a pool the library keeps, with
 * non-temporal stores (cached_stores == 0: the array is larger than the host's caches and is written once) or ordinary
 * stores (cached_stores != 0: the consumer reads it right away and it fits the last-level cache). All pointers are HOST pointers; adj must be 16-byte aligned (4-byte when E*E % 4 != 0). Pure data movement - every float is
 * either copied or zero. */
int lsm_expand_adjacency_host(const float *adj_base, const uint32_t *adj_keep, float *adj, int64_t num_envs,
                              int32_t num_agents, int32_t num_entities, int32_t threads, int32_t cached_stores);

/* HOST buffers of one reference-facing step (GraphSubprocVecEnv.step_wait returns host arrays,
 * onpolicy/envs/env_wrappers.py:983-996). Every pointer is a HOST pointer; page-locked memory makes the copies true DMA.
 * NULL = that array is not fetched (adj and the two staging arrays are required). */
typedef struct lsm_host_io {
    float *obs;               /* [num_envs][N][D]        */
    float *node_obs;          /* [num_envs][N][E][F]     (F = 7 with graph_feat_type='global') */
    float *adj;               /* [num_envs][N][E][E]     dense, rebuilt on the host; pageable memory is fine */
    float *reward;            /* [num_envs][N]           */
    uint8_t *done;            /* [num_envs][N]           */
    float *adj_base_staging;  /* [num_envs][E][E]        landing area of the compact adjacency (page-locked) */
    uint32_t *adj_keep_staging; /* [num_envs][N][W]      W = ceil(E / 32) */
    int32_t threads;          /* host worker threads of the expansion (<= 0: one per online core, at most 16) */
    int32_t chunks;           /* env ranges the adjacency crosses PCIe in (<= 0: automatic) */
    int32_t cached_stores;    /* see lsm_expand_adjacency_host */
    int32_t reserved;
} lsm_host_io;

/* Device -> host of the CURRENT outputs with the compact adjacency active (lsm_set_compact_adjacency): the thresholded
 * matrices + keep masks leave first in `chunks` env ranges, the library's host threads expand each range into io->adj as
 * it lands while the DMA engine is still moving the later ranges and node_obs / obs / reward / done. Returns when every
 * host array is complete (the stream's work up to this call has finished). */
int lsm_fetch_host(lsm_handle *h, const lsm_host_io *io, void *stream);

/* The whole reference-facing step with HOST buffers in ONE call - what a host-language binding of
 * GraphSubprocVecEnv.step(actions) (env_wrappers.py:951-996, 103-110) calls: actions host -> device (exactly one of the
 * two HOST action arrays: int32 [num_envs][N] indices or float32 [num_envs][N][25] one-hot rows; page-locked memory is
 * DMA'd in place, pageable memory is staged), lsm_step, lsm_fetch_host. */
int lsm_step_host(lsm_handle *h, const int32_t *action_idx_host, const float *action_onehot_host, int64_t episode,
                  uint64_t seed, int auto_reset, const lsm_host_io *io, void *stream);

/* Compacted COO edge list of the adjacency output in the order the reference's GNN builds on every forward
 * (TransformerConvNet.process_adj, onpolicy/algorithms/utils/gnn.py:376-407): graphs = num_envs * N, row-major
 * non-zeros of each E x E matrix;
 *   edge_index  DEVICE int64 [2][capacity]: row 0 = graph * E + row, row 1 = graph * E + col
 *   edge_attr   DEVICE float [capacity]
 *   counts      DEVICE int32 [graphs]         non-zeros per graph
 *   offsets     DEVICE int64 [graphs + 1]     exclusive prefix sum; offsets[graphs] = nnz (entries past `capacity`
 *                                             are not written - check nnz <= capacity)
 * adj = NULL reads the bound adj output of the last step. */
int lsm_edge_list(lsm_handle *h, const float *adj, int64_t *edge_index, float *edge_attr, int32_t *counts,
                  int64_t *offsets, int64_t capacity, void *stream);

/* Fused edge output (SURVEY 8f N2): from now on every lsm_step / lsm_reset / lsm_observe ALSO writes the COO list of
 * the step's adjacency, in the same order and layout as lsm_edge_list, straight from the emission kernel (row masks by
 * ballot, ranks by popcount, per-graph start offsets from a counting pre-pass over the per-env records) - the dense
 * tensor is not read back, and with dense_adj == 0 it is not written at all (the 4*N*E*E term of SURVEY 8d disappears;
 * per edge 20 bytes are written instead, which pays when the mean degree is below ~E/5). Nothing is synchronised:
 * offsets[graphs] holds nnz ON THE DEVICE; entries past `capacity` are dropped (counts, offsets and nnz stay exact).
 * A masked lsm_reset writes the list of ALL environments, the ones outside the mask from their unchanged state; this
 * holds for the first launch after this call too (the arrays need no prior contents). All four pointers NULL switches
 * it off. Specialised (dynamics, N, L) configurations only, in either interpolation mode (returns 6 otherwise).
 *   edge_index DEVICE int64 [2][capacity], edge_attr DEVICE float [capacity], counts DEVICE int32 [graphs],
 *   offsets DEVICE int64 [graphs + 1]                                         graphs = num_envs * N */
int lsm_set_edge_output(lsm_handle *h, int64_t *edge_index, float *edge_attr, int32_t *counts, int64_t *offsets,
                        int64_t capacity, int dense_adj);

/* The renderer's world graph (SURVEY 8a a16): SafeAamScenario.update_graph, navigation_graph_safe.py:996-1015, as
 * MultiAgentGraphEnv.step would compute it at the top of the NEXT step (environment.py:964-965) from the bound state:
 * one graph per environment over its E entities, entities that are disconnected (agent done / landmark already reached)
 * removed, an edge wherever 0 < d <= max_edge_dist (INCLUSIVE radius, unlike the policy-facing adjacency), row-major.
 *   edge_index  DEVICE int64 [2][capacity]: row 0 = entity row, row 1 = entity col (indices inside the environment)
 *   edge_weight DEVICE double [capacity]    the distance (world.edge_weight)
 *   counts      DEVICE int32 [num_envs], offsets DEVICE int64 [num_envs + 1] (offsets[num_envs] = nnz) */
int lsm_world_graph(lsm_handle *h, int64_t *edge_index, double *edge_weight, int32_t *counts, int64_t *offsets,
                    int64_t capacity, void *stream);

/* Rollout-buffer bookkeeping of one step in one launch (reference GMPERunner.insert + GraphReplayBuffer.insert,
 * onpolicy/runner/shared/graph_mpe_runner.py:437-487, onpolicy/utils/graph_buffer.py:168-250), all DEVICE pointers:
 *   obs           float [num_envs][N][D]       the observation slot the step kernels just wrote
 *   done          uint8 [num_envs][N]          the step's done flags
 *   share_obs     float [num_envs][N][N*D]     <- every agent's obs of the env, concatenated (NULL: not centralised)
 *   masks         float [num_envs][N]          <- 0 where done else 1
 *   active_masks  float [num_envs][N]          <- like masks, but 1 for every agent of an env whose agents are all done */
int lsm_rollout_insert(lsm_handle *h, const float *obs, const uint8_t *done, float *share_obs, float *masks,
                       float *active_masks, void *stream);

/* Episode statistics of this shard for the runner's log line (MultiAgentGraphEnv.reset's summary dict, multiagent/environment.py:
 * 1065-1073, averaged over the vectorised envs at onpolicy/runner/shared/graph_mpe_runner.py:155-158): out = DEVICE double
 * [LSM_EP_COUNT + 1], the SUM over the bound environments of every column of ep_info followed by the environment count - the 9
 * doubles a multi-GPU job all-reduces at log time (the only collective of the path). One launch, no host sync, fixed order. */
int lsm_episode_stats(lsm_handle *h, double *out, void *stream);

/* The float64 sin / cos / atan2 of include/lsm_math.h (what the kernels use instead of libdevice so that they agree bit
 * for bit with the CPU oracle), evaluated on the HOST (lsm_math_eval: a, b, out are host pointers; no GPU needed -
 * B200GraphVecEnv.set_state tabulates the landmark heading sin / cos with it, like the on-device reset does) or on the
 * DEVICE (lsm_math_eval_device: device pointers). op: 0 sin(a), 1 cos(a), 2 atan2(a, b), 3 / 4 the sin / cos half of the
 * header's one-reduction sincos; b may be NULL unless op == 2. Replaces numpy's libm at multiagent/core.py:105-131,179-181,
 * safety_filter.py:277-284, navigation_graph_safe.py:606-656, utils.py:79-349. */
int lsm_math_eval(int op, const double *a, const double *b, double *out, int64_t n);
int lsm_math_eval_device(int op, const double *a, const double *b, double *out, int64_t n, void *stream);

/* Tell the library that the caller edited the bound state tensors (agent_f64 / agent_i32 / env_f64) directly.
 * The specialised pipeline keeps the HJ pair values of the current state from the previous launch
 * (safety_filter.py:192-201 evaluated one step ahead); after an edit the next lsm_step recomputes them first. */
int lsm_invalidate(lsm_handle *h);

/* Measurement hook (specialised pipeline only): relaunch the graph-emission kernel alone on the per-env
 * records the last lsm_step / lsm_reset / lsm_observe left behind. Idempotent: rewrites node_obs and adj
 * (graph_observation, navigation_graph_safe.py:932-994) with the same values. Returns 6 when the
 * configuration has no separate emission launch. */
int lsm_emit_only(lsm_handle *h, void *stream);

/* Rollout storage by emit record (specialised pipeline only). The graph observation of one environment at one step is a
 * pure function of its emit record (emit_record_bytes of lsm_launch_info, 1-7 % of the dense node_obs + adj bytes) and
 * of the handle's constants (radius, graph_feat_type), so a rollout can keep the records and rebuild any observer's
 * graph when a learner asks for it.
 *
 * lsm_copy_records: copy the num_envs * emit_record_bytes records that the last lsm_step / lsm_reset / lsm_observe left
 * behind to `dst` (device or pinned host memory) with one cudaMemcpyAsync on `stream`. After a masked reset the envs
 * outside the mask keep the record of their previous step, which is also what their node_obs / adj still hold. Returns
 * 6 on a generic-kernel handle, 5 when no buffers are bound. */
int lsm_copy_records(lsm_handle *h, void *dst, void *stream);

/* lsm_emit_from_records: for each item k, the node rows and the masked thresholded adjacency matrix that observer
 * observer[k] received at the step of record record[k], byte for byte what the step's emission wrote to its node_obs /
 * adj. Uses the handle's shape, graph_feat_type and coordination_range; needs no bound buffers, launches on `stream`
 * and never synchronises. An item whose record is outside [0, num_records) or whose observer is outside [0, N) gets
 * zero-filled outputs. Returns 6 on a generic-kernel handle. */
typedef struct lsm_record_emit_io {
    int64_t num_items;          /* B >= 0 */
    int64_t num_records;        /* records in the store */
    const void *records;        /* DEVICE [num_records][emit_record_bytes], 16-byte aligned, written by lsm_copy_records
                                   of a handle of the same library and shape */
    const int64_t *record;      /* DEVICE [B] */
    const int32_t *observer;    /* DEVICE [B] */
    float *node_obs;            /* DEVICE [B][E][F] out (F = 7 with graph_feat_type global), 16-byte aligned, or NULL */
    float *adj;                 /* DEVICE [B][E][E] out, 16-byte aligned, or NULL */
} lsm_record_emit_io;
int lsm_emit_from_records(lsm_handle *h, const lsm_record_emit_io *io, void *stream);

/* lsm_edges_from_records: the COO edge list of the matrices lsm_emit_from_records would write for the same items, in the
 * order and layout of the reference's TransformerConvNet.process_adj (gnn.py:376-407) over the (B, E, E) batch: item k's
 * non-zero entries in row-major order, edge_index row 0 = k * E + row, row 1 = k * E + col, edge_attr = the matrix entry
 * bit for bit. No dense matrix is written or read. Two passes over the same items:
 *   edge_index == NULL  counting pass: writes counts and offsets (exclusive prefix, offsets[B] = nnz on the device).
 *                       Zero items: only offsets[0] = 0.
 *   otherwise           fill pass: reads the offsets of a counting pass and writes only positions in [0, capacity), so a
 *                       short capacity or a stale offsets array never writes out of bounds. Zero items: nothing.
 * Items with an out-of-range record or observer have no edges. Uses the handle's shape and coordination_range, needs no
 * bound buffers, keeps no per-handle scratch, launches on `stream` and never synchronises (two streams may use one
 * handle at once). Returns 6 on a generic-kernel handle, 2 on negative sizes, missing arrays or misaligned records. */
typedef struct lsm_record_edges_io {
    int64_t num_items;          /* B >= 0 */
    int64_t num_records;        /* records in the store */
    const void *records;        /* as lsm_record_emit_io */
    const int64_t *record;      /* DEVICE [B] */
    const int32_t *observer;    /* DEVICE [B] */
    int32_t *counts;            /* DEVICE [B]   edges per item (counting pass) */
    int64_t *offsets;           /* DEVICE [B+1] offsets[B] = nnz (written by the counting pass, read by the fill pass) */
    int64_t *edge_index;        /* DEVICE [2][capacity], or NULL (counting pass) */
    float *edge_attr;           /* DEVICE [capacity] */
    int64_t capacity;
} lsm_record_edges_io;
int lsm_edges_from_records(lsm_handle *h, const lsm_record_edges_io *io, void *stream);

/* Diagnostics (never on the product path): per-kernel timeline of the launches that follow. If `out_ns` is non-NULL
 * and a timeline is armed, synchronises the device and copies 7 %globaltimer values (ns) out: pair first-block-in,
 * pair last-body-out, agent in / out, emit in / out, pair grid out. `arm` != 0 (re)arms the recording for the next
 * launches, 0 disables it. */
int lsm_debug_timeline(lsm_handle *h, int arm, uint64_t *out_ns);

/* Diagnostics (never on the product path): copy the specialised pipeline's HJ pair-value scratch, the raw values
 * V(x_i - x_j) the next lsm_step's filter starts from, to `out` (device or pinned host memory, num_envs * N * N
 * doubles, [env][ego][other]) with one cudaMemcpyAsync on `stream`. Read-only. Only the entries the next step reads
 * are defined: envs whose curriculum has the filter on, i != j, both agents not done. Returns 6 when the
 * configuration keeps no pair values (generic kernel). */
int lsm_debug_pair_values(lsm_handle *h, double *out, void *stream);

/* The HJ safety filter as a standalone batched operator, for states the environment does not own (another simulator,
 * hardware, logged trajectories). Both entry points need a handle with a value grid (lsm_set_value_grid); buffers need
 * not be bound. They use the handle's dynamics, grid, interpolation mode (LSM_FLAG_INTERP_FLOAT32) and its config's dt,
 * cbf_rate and coordination_range, evaluate the relative state in the form of the specialised pipeline (one sincos of
 * the ego heading per pair), launch on `stream` and never synchronise. All pointers are DEVICE pointers; states are
 * double integrator [x, y, vx, vy] or airtaxi [x, y, theta, v]; d = 4 (double integrator) | 5 (airtaxi).
 *
 * lsm_safety_filter: the safety handle's apply_safety_filter (safety_filter.py:203-260, 378-433) for num_rows
 * independent egos, each against num_slots candidate others. Per row: distance and HJ value of every active slot, the
 * FIRST minimum of each in ascending slot order (np.argmin), the value shifted by -(sep - grid separation), then the
 * range test against coordination_range, gradient, bang-bang below 0.4 or CBF-QP, clipping and
 * filtered = |u - u_ref| > 1e-4, exactly as lsm_step computes it for one ego. index is the deconflicting slot, also when
 * the row stays unfiltered because of range; -1 and value +inf when no slot is active. If every active value is +inf
 * (NaN state) index is the first active slot, value +inf and the row is unfiltered. */
typedef struct lsm_filter_io {
    int64_t num_rows;                   /* B >= 0 */
    int32_t num_slots;                  /* M >= 0 */
    int32_t _reserved;
    const double *ego;                  /* [B][4] */
    const double *others;               /* [B][M][4] (may be NULL when M == 0) */
    const double *ego_action;           /* [B][2]    decoded control of the ego */
    const double *other_actions;        /* [B][M][2] decoded reference controls of the others (may be NULL when M == 0) */
    const uint8_t *active;              /* [B][M] slot mask (0 = absent) or NULL = every slot active */
    const double *separation_distance;  /* [B] or NULL = the grid's own separation (no shift) */
    double *safe_action;                /* [B][2] out */
    uint8_t *filtered;                  /* [B] out, or NULL */
    int32_t *index;                     /* [B] out, or NULL */
    double *value;                      /* [B] out, or NULL */
} lsm_filter_io;
int lsm_safety_filter(lsm_handle *h, const lsm_filter_io *io, void *stream);

/* lsm_hj_lookup: get_value_of_relative_state (safety_filter.py:192-201, 345-354) and the gradient (:245, :418) for
 * num_points points, given as relative states (rel non-NULL) or as (ego, other) state pairs. value: +inf for a NaN
 * relative state, shifted like the filter's; a finite point outside the grid box is interpolated with the grid's index
 * clamp, as the env does. grad: every component NaN for a NaN relative state. */
typedef struct lsm_lookup_io {
    int64_t num_points;                 /* K >= 0 */
    const double *rel;                  /* [K][d] or NULL: then ego / other */
    const double *ego;                  /* [K][4] */
    const double *other;                /* [K][4] */
    const double *separation_distance;  /* [K] or NULL = the grid's own separation */
    double *value;                      /* [K] out */
    double *grad;                       /* [K][d] out, or NULL */
    double *rel_out;                    /* [K][d] out: the relative state used, or NULL */
} lsm_lookup_io;
int lsm_hj_lookup(lsm_handle *h, const lsm_lookup_io *io, void *stream);

#ifdef __cplusplus
}
#endif
#endif
