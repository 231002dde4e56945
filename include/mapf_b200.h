/*
 * mapf_b200.h -- C ABI of libmapf_b200.so: the batched, B200-native (sm_100a) implementation
 * of the MAPF environment transition of Nerozud/dl_reference_models.
 *
 * Reference interface replaced (ENV = src/environments/reference_model_multi_agent.py):
 *   ReferenceModel.__init__(env_config)   ENV:34-193   -> mapf_create + mapf_set_map + mapf_bind_state
 *   ReferenceModel.reset()                ENV:440-472  -> mapf_reset / mapf_reset_host
 *   ReferenceModel.step(action_dict)      ENV:474-695  -> mapf_step  / mapf_step_host
 *   get_obs / get_action_mask             ENV:707-773  -> the local_obs / action_mask outputs
 *   _flatten_observation                  ENV:306-328  -> mapf_pack_flat_obs
 *   private state arrays (ENV:82-120), written by the reference's tests -> mapf_state tensors
 *   info["__all__"] + RLlib callback metric set (src/trainers/callbacks.py:152,173,335-345)
 *                                                       -> env_words / mapf_metrics_reduce
 *
 * Conventions
 *   - plain C: opaque handle, plain pointers and sizes, every call returns 0 or a negative
 *     MAPF_ERR_* code; mapf_last_error() gives the message (thread-local).  No exceptions.
 *   - one handle <-> one CUDA device; a handle is not thread-safe.
 *   - B = num_envs on this device, N = num_agents (<= 32), V = 2*sensor_range+1 (sr <= 3),
 *     coordinates are (row, col) int16 pairs like the reference's int16 [N,2] arrays.
 *   - `stream` arguments are cudaStream_t passed as void* (NULL = legacy default stream).
 *   - "device pointer" buffers are caller-owned (e.g. torch tensors); *_host entry points take
 *     host pointers and do the H2D / D2H copies themselves on the handle's own stream (pass
 *     page-locked buffers for full PCIe/NVLink-C2C bandwidth; pageable memory works too).
 *   - there is NO CPU fallback: every entry point that computes launches sm_100a kernels.
 */
#ifndef MAPF_B200_H
#define MAPF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAPF_MAX_AGENTS 32
#define MAPF_MAX_SENSOR_RANGE 3
#define MAPF_MAX_LOCK_WINDOW 32
#define MAPF_MAX_DIM 255

#define MAPF_OK 0
#define MAPF_ERR_INVALID_ARG (-1)
#define MAPF_ERR_CUDA (-2)
#define MAPF_ERR_UNSUPPORTED (-3)
#define MAPF_ERR_STATE (-4)

/* device-side error bits, see mapf_poll_errors() */
#define MAPF_DEV_ERR_INVALID_ACTION 1u /* ENV:504-506 (ValueError in the reference) */
#define MAPF_DEV_ERR_NO_GOAL_CELL 2u   /* ENV:296-298 (RuntimeError in the reference) */
#define MAPF_DEV_ERR_TOO_FEW_CELLS 4u  /* ENV:270-275 (ValueError in the reference) */
#define MAPF_DEV_ERR_DUPLICATE_LAYOUT 8u /* a starts / goals override names one cell twice (a layout is 2N distinct cells, ENV:277) */

/* env_config keys that affect the transition (ENV:38-61), plus batching/sharding keys. */
typedef struct mapf_config {
    int32_t num_envs;    /* B: envs owned by this handle (this GPU's shard) */
    int32_t num_agents;  /* N, 1..32 */
    int32_t rows, cols;  /* map shape, 1..255 */
    int32_t sensor_range;      /* 1..3 */
    int32_t steps_per_episode; /* ENV:38 */
    int32_t lifelong_mapf;     /* ENV:51 */
    int32_t enable_lock_metrics;   /* ENV:61 */
    int32_t deadlock_window_steps; /* ENV:56, 1..32 */
    int32_t livelock_window_steps; /* ENV:57, 1..32 */
    int32_t lock_nearby_manhattan; /* ENV:58 */
    int32_t lock_min_neighbors;    /* ENV:60 */
    int32_t lock_progress_epsilon_floor; /* floor(ENV:59): distances are integers */
    int32_t normalize_goal_delta;  /* ENV:42 */
    int32_t deterministic;   /* ENV:41: reset restores `starts`, keeps goals (ENV:452-455) */
    int32_t per_env_maps;    /* 0: one map shared by all envs; 1: one map per env */
    int64_t env_id_base;     /* global id of env 0 (Philox key => results independent of sharding) */
    uint64_t seed;           /* ENV:74 */
    int32_t device;          /* CUDA device ordinal */
    int32_t step_kernel;     /* 0 auto, 1 lane-per-agent kernel, 2 env-per-thread kernel (cols <= 32, shared map), 3 two lanes per env (same limits, num_agents % 4 == 0) */
} mapf_config;

/* Words of the per-env int32 state block env_words[B, MAPF_ENV_WORDS]. */
enum {
    MAPF_W_STEP_COUNT = 0,      /* ENV:37 */
    MAPF_W_LOCK_COUNT,          /* ENV:119 _lock_hist_count, not saturated: history rows appended since reset */
    MAPF_W_LOCK_PREV,           /* bit0 _deadlock_state_prev, bit1 _livelock_state_prev (ENV:68-69) */
    MAPF_W_GOALS_TOTAL,         /* ENV:88  _episode_goals_reached_total */
    MAPF_W_BLOCKING_TOTAL,      /* ENV:63  _episode_blocking_count */
    MAPF_W_DEADLOCK_EVENTS,     /* ENV:64 */
    MAPF_W_LIVELOCK_EVENTS,     /* ENV:65 */
    MAPF_W_DEADLOCK_STEPS,      /* ENV:66 */
    MAPF_W_LIVELOCK_STEPS,      /* ENV:67 */
    MAPF_W_RNG_COUNTER,         /* Philox draws consumed by this env */
    MAPF_W_EPISODE_RETURN_X2,   /* 2 * sum of rewards of all agents this episode (exact integer) */
    MAPF_W_WFG_CYCLE_STEPS,     /* steps of this episode with a wait-for-graph cycle */
    MAPF_W_EPISODES,            /* finished episodes of this env */
    MAPF_W_LOCK_HEAD,           /* ENV:120 _lock_hist_head of the distance ring (slot of the next row) */
    MAPF_W_RESERVED1,
    MAPF_W_RESERVED2,
    MAPF_ENV_WORDS
};

/* agent_flags bits (state tensor agent_flags[B,N], uint8) */
#define MAPF_AF_REACHED 1u        /* ENV:86 _reached_arr (sticky) */
#define MAPF_AF_COMPLETED_ONCE 2u /* ENV:87 _completed_once_arr */
#define MAPF_AF_BLOCKING_PREV 4u  /* ENV:89 _blocking_pressure_prev_arr (as 0/1) */
/* ENV:102 _occupancy_owner, the part positions do not determine: the agent stands on a cell it does not own.
 * Never set by a legal step (ENV:516-521 keeps agents apart); only after several agents were injected onto one
 * cell (the states ENV:658-666 penalises): the highest index owns the cell (ENV:200-205), a leaving agent clears
 * the owner for everybody (ENV:523).  Honoured and maintained by the env-per-thread step kernel. */
#define MAPF_AF_NOT_OWNER 8u

/* Device-resident state, caller-owned (torch tensors).  Layout mirrors ENV:82-120. */
typedef struct mapf_state {
    int16_t *positions;    /* [B,N,2] ENV:84 */
    int16_t *goals;        /* [B,N,2] ENV:85 */
    int16_t *starts;       /* [B,N,2] ENV:83 */
    uint8_t *agent_flags;  /* [B,N]   MAPF_AF_* */
    uint32_t *lock_goal_progress; /* [B,N] bit t = flag t steps ago (ENV:115) */
    uint32_t *lock_moved;         /* [B,N] (ENV:116) */
    uint32_t *lock_failed_move;   /* [B,N] (ENV:117) */
    int16_t *lock_distance;       /* [B,LW,N] ring over the livelock window (ENV:118) */
    int32_t *env_words;    /* [B,MAPF_ENV_WORDS] */
    double *env_metrics;   /* [B,MAPF_METRIC_COUNT] per-env episode-end sums (see below) */
} mapf_state;

/* Episode-end metric sums (the set the reference's RLlib callbacks log,
 * src/trainers/callbacks.py:152,173,335-345).  Per env in env_metrics, reduced by
 * mapf_metrics_reduce(); ranks all-reduce(sum) the reduced vector. */
enum {
    MAPF_M_EPISODES = 0,
    MAPF_M_RETURN_SUM,
    MAPF_M_LENGTH_SUM,
    MAPF_M_SUCCESS_SUM,      /* terminated && !truncated, callbacks.py:172 */
    MAPF_M_GOALS_REACHED_SUM,
    MAPF_M_BLOCKING_COUNT_SUM,
    MAPF_M_DEADLOCK_COUNT_SUM,
    MAPF_M_LIVELOCK_COUNT_SUM,
    MAPF_M_DEADLOCK_STEPS_SUM,
    MAPF_M_LIVELOCK_STEPS_SUM,
    MAPF_M_THROUGHPUT_SUM,
    MAPF_M_COMPLETION_RATIO_SUM,
    MAPF_M_WFG_CYCLE_STEPS_SUM,
    MAPF_M_RESERVED0,
    MAPF_M_RESERVED1,
    MAPF_M_RESERVED2,
    MAPF_METRIC_COUNT
};

/* step_flags bits (output step_flags[B], uint8) */
#define MAPF_SF_TERMINATED 1u      /* ENV:675,686 */
#define MAPF_SF_TRUNCATED 2u       /* ENV:687 */
#define MAPF_SF_DEADLOCK_STEP 4u   /* ENV:644 */
#define MAPF_SF_LIVELOCK_STEP 8u   /* ENV:645 */
#define MAPF_SF_DEADLOCK_EVENT 16u /* ENV:646 */
#define MAPF_SF_LIVELOCK_EVENT 32u /* ENV:647 */
#define MAPF_SF_GOAL_REASSIGNED 64u /* ENV:556 */
#define MAPF_SF_WFG_CYCLE 128u     /* wait-for-graph cycle present (no reference counterpart) */

/* agent_step_flags bits (output agent_step_flags[B,N], uint8) */
#define MAPF_ASF_MOVED 1u          /* ENV:582 */
#define MAPF_ASF_FAILED_MOVE 2u    /* ENV:583 */
#define MAPF_ASF_GOAL_REACHED 4u   /* info[aid]["goal_reached_step"], ENV:629 */
#define MAPF_ASF_BLOCKING 8u       /* info[aid]["blocking"], ENV:628 */
#define MAPF_ASF_WFG_CYCLE 16u     /* agent is on a wait-for-graph cycle */
#define MAPF_ASF_ON_GOAL 32u       /* ENV:588 current_on_goal */

/* Outputs of reset/step.  Caller-owned; any pointer may be NULL (that channel is skipped). */
typedef struct mapf_outputs {
    uint8_t *local_obs;     /* [B,N,V,V] ENV:707-747 (staggered snapshot, F3) */
    int8_t *action_mask;    /* [B,N,5]   ENV:749-773 */
    float *goal_delta;      /* [B,N,2]   ENV:330-335 */
    uint8_t *blocking_prev; /* [B,N]     ENV:322 (0/1) */
    float *reward;          /* [B,N] */
    uint8_t *terminated;    /* [B] */
    uint8_t *truncated;     /* [B] */
    uint8_t *step_flags;        /* [B]   MAPF_SF_* */
    uint8_t *agent_step_flags;  /* [B,N] MAPF_ASF_* */
    int32_t *info;              /* [B,MAPF_INFO_WORDS] integer sources of info["__all__"], ENV:639-656 */
} mapf_outputs;

/* Words of the per-step info block (all exact integers; the two ratios of ENV:638,655 are
 * completed_count / N and goals_reached_total / max(step_count, 1), formed by the caller in
 * float64 like the reference does). */
enum {
    MAPF_I_GOALS_REACHED_STEP = 0,
    MAPF_I_GOALS_REACHED_TOTAL,   /* lifelong: cumulative arrivals, else sum(_reached_arr), ENV:630-633 */
    MAPF_I_BLOCKING_COUNT_STEP,
    MAPF_I_BLOCKING_COUNT_TOTAL,
    MAPF_I_DEADLOCK_STEP,
    MAPF_I_LIVELOCK_STEP,
    MAPF_I_DEADLOCK_EVENT_STEP,
    MAPF_I_LIVELOCK_EVENT_STEP,
    MAPF_I_DEADLOCK_EVENTS_TOTAL,
    MAPF_I_LIVELOCK_EVENTS_TOTAL,
    MAPF_I_DEADLOCK_STEPS_TOTAL,
    MAPF_I_LIVELOCK_STEPS_TOTAL,
    MAPF_I_COMPLETED_COUNT,       /* sum(_completed_once_arr), ENV:638 */
    MAPF_I_STEP_COUNT,            /* ENV:655 */
    MAPF_I_REACHED_COUNT,         /* sum(_reached_arr) */
    MAPF_I_WFG_CYCLE_STEPS,
    MAPF_INFO_WORDS
};

typedef struct mapf_handle mapf_handle;

const char *mapf_version(void);
const char *mapf_last_error(void);

/* ENV:34-193.  Validates cfg (limits above), allocates the handle's small device tables. */
int mapf_create(const mapf_config *cfg, mapf_handle **out);
int mapf_destroy(mapf_handle *h);

/* grid: HOST uint8 [R,C] (shared) or [B,R,C] (per_env_maps), 0 free / 1 obstacle (ENV:80-82).
 * Returns MAPF_ERR_INVALID_ARG if a map has fewer than 2N free cells and cfg is not
 * deterministic (ENV:270-275). */
int mapf_set_map(mapf_handle *h, const uint8_t *grid);

/* Bytes the caller must allocate for each mapf_state member (same order as the struct). */
int mapf_state_nbytes(const mapf_handle *h, int64_t out_nbytes[10]);
/* Install the device pointers of the state tensors (kept by reference, not copied). */
int mapf_bind_state(mapf_handle *h, const mapf_state *state);
/* Alternative for callers without their own device allocator (plain C / cgo / ctypes users):
 * the handle allocates, zeroes, binds and later frees the state block itself. */
int mapf_alloc_state(mapf_handle *h);
/* Copy the bound state device -> host / host -> device.  `host` holds HOST pointers with the
 * mapf_state layout; NULL members are skipped.  This is the injection path the reference's
 * tests use by writing the private numpy arrays (tests/test_reference_model_lifelong.py:29-39). */
int mapf_get_state_host(mapf_handle *h, const mapf_state *host);
int mapf_set_state_host(mapf_handle *h, const mapf_state *host);

/* ENV:440-472.  reset_mask: device uint8 [B] (NULL = every env).
 * starts_override / goals_override: device int16 [B,N,2] or NULL.  With overrides the layout is
 * taken from them (what rng.choice produced, ENV:277-280); otherwise deterministic cfg restores
 * `starts`, and non-deterministic cfg draws 2N distinct free cells with Philox4x32-10
 * keyed by (seed, env_id_base + env). */
int mapf_reset(mapf_handle *h, const uint8_t *reset_mask, const int16_t *starts_override,
               const int16_t *goals_override, const mapf_outputs *out, void *stream);

/* ENV:707-773 on the CURRENT state (the public get_obs()/get_action_mask() of the reference):
 * fills local_obs / action_mask / goal_delta / blocking_prev of `out`, mutates nothing. */
int mapf_observe(mapf_handle *h, const mapf_outputs *out, void *stream);
int mapf_observe_host(mapf_handle *h, const mapf_outputs *out_host);

/* ENV:474-695.  actions: device int8 [B,N] in 0..4 (NULL = all NO_OP, ENV:498-500).
 * goal_override: device int16 [B,N,2]; a row >= 0 replaces the lifelong goal draw of that agent
 *   (replay hook for bit-exact parity; NULL = none).
 * goal_rank: device int32 [B,N]; a value >= 0 replaces rng.integers(n) at ENV:300 (NULL = none).
 * auto_reset != 0: an env whose episode ended is reset in the same launch (its obs outputs are
 *   the first observation of the next episode; reward/terminated/truncated are the final step's),
 *   like run_benchmark's `if done: reset()` (scripts/benchmark_multi_agent_env.py:89-95). */
int mapf_step(mapf_handle *h, const int8_t *actions, const int16_t *goal_override,
              const int32_t *goal_rank, const mapf_outputs *out, int32_t auto_reset, void *stream);

/* `steps` consecutive env steps in one call, for rollouts whose actions come from the fused benchmark sampler
 * (mapf_set_fused_sampler; scripts/benchmark_multi_agent_env.py:38-57): step 1 takes `actions`, step t + 1 the
 * actions drawn at the end of step t -- exactly what `steps` calls of mapf_step would do, bit for bit, but inside ONE
 * kernel launch (lane-per-agent and env-per-thread kernels; the two-lanes-per-env kernel launches `steps` times): small
 * batches stop being launch-rate bound (~10 us per launch for 4 096 x 4), GPU-filling ones pay ramp-up and tail once
 * and read each step's state from L2 -- every warp takes its envs from the first step to the last.
 * Step t writes its outputs t * out_step_stride_envs envs further into `out` (pass [steps, B, ...] buffers and
 * stride B for a rollout, or 0 to keep only the last step's).  The sampler's action buffer holds the actions for
 * the step after the last.  No replay hooks (goal_override / goal_rank) on this entry point. */
int mapf_step_many(mapf_handle *h, const int8_t *actions, const mapf_outputs *out, int32_t steps,
                   int64_t out_step_stride_envs, int32_t auto_reset, void *stream);

/* Host-buffer variants: same semantics, every pointer is HOST memory (NULL = skip).
 * H2D of inputs, the kernel, and D2H of the requested outputs all happen inside the call,
 * which returns after the results are in the host buffers. */
int mapf_reset_host(mapf_handle *h, const uint8_t *reset_mask, const int16_t *starts_override,
                    const int16_t *goals_override, const mapf_outputs *out_host);
/* STREAM ORDER of the *_host entry points.  They run on two private non-blocking streams of the handle and are
 * synchronous: when they return, their results are in the host buffers and the device state is final, so anything
 * queued AFTER them (on any stream) is ordered.  For work queued BEFORE them the rule is: everything enqueued
 * through this handle's stream-taking entry points (mapf_reset / mapf_step / mapf_observe / samplers / flat pack)
 * is waited for automatically -- the handle remembers the last such stream and makes its private streams wait on
 * an event recorded there.  Work the library cannot see (a caller's own kernels or copies into the bound state
 * tensors, e.g. torch ops) must be announced with mapf_host_wait_stream(h, stream) before the next *_host call;
 * BatchedMapfEnv.step_host / reset_host do that with torch's current stream.  mapf_set_state_host /
 * mapf_get_state_host synchronise the whole device before and their own copies after: on return the state is on
 * the device (resp. in the host arrays) even when the host arrays are pageable. */
int mapf_host_wait_stream(mapf_handle *h, void *stream);
int mapf_step_host(mapf_handle *h, const int8_t *actions, const int16_t *goal_override,
                   const int32_t *goal_rank, const mapf_outputs *out_host, int32_t auto_reset);

/* mapf_step_host is PCIe-bound on big batches.  When local_obs, action_mask, goal_delta and reward are all
 * requested (and num_envs >= 8192, rows/cols <= 128) those channels cross PCIe as one bit-packed record per
 * agent (3 bits per window cell, 1 bit per mask entry, the integer goal difference, 2*reward) and host threads
 * inside the call expand them into the caller's arrays -- the delivered arrays are bit for bit the same.
 * Whether it pays depends on the host (PCIe rate against what its cores and memory system can expand, with
 * whatever else -- the other ranks of a multi-GPU node -- runs beside it), so the handle measures: its first sixteen
 * eligible calls go four at a time -- a warm-up, then packed, packed with a non-temporal expansion (cache-resident blocks streamed out as
 * whole lines: no read-for-ownership of the arrays, which is what counts on a host bound by its memory system), plain;
 * the first of each four untimed, the best of the other three counts -- and the fastest mode stays (in that order of
 * preference: a later one has to win by 10 %); ranks that share a node should make these calls
 * in step, so that each of them measures the host it will run on.  MAPF_HOST_PACK=0 / 1 and MAPF_HOST_NT=0 / 1 force the
 * choices, MAPF_HOST_THREADS / MAPF_HOST_SLICES tune it.  The expansion
 * threads (cores of this process / LOCAL_WORLD_SIZE, at most 16, the caller's thread included) are pinned one per
 * core to this rank's chunk of the affinity mask when the node is shared (MAPF_HOST_PIN=0 / 1 overrides).
 * mapf_host_transfer_bytes: bytes that actually crossed PCIe in the last mapf_step_host call. */
int mapf_host_transfer_bytes(const mapf_handle *h, int64_t *h2d_bytes, int64_t *d2h_bytes);
/* How mapf_step_host delivers the four big channels on this handle: -1 still measuring (its first sixteen eligible calls
 * try each mode), 0 plain copies, 1 bit-packed + expansion by host threads, 2 the same with the expansion going through
 * cache-resident blocks and non-temporal stores (hosts bound by their memory system).  MAPF_HOST_PACK / MAPF_HOST_NT
 * force a mode. */
int mapf_host_transfer_mode(const mapf_handle *h);
/* Compact delivery, for callers that accept it: local_obs, action_mask, goal_delta and reward arrive as the
 * bit-packed records themselves -- `records_host` (pinned recommended) receives, for the whole batch of BN = B * N
 * agents, [BN x mapf_packed_record_bytes(v2) - 3 bytes: window + mask bits][BN x (int8 d_row, int8 d_col)][BN x int8
 * 2*reward], i.e. exactly the block mapf_unpack_records expands -- and nothing is expanded inside the call: 13 B per
 * agent cross PCIe and reach host memory instead of 42 B.  A consumer expands what it needs when it needs it (a
 * learner, per minibatch) with mapf_unpack_records, bit for bit the arrays mapf_step_host would have delivered.
 * `out_host_small`: the remaining channels (blocking_prev, terminated, truncated, step_flags, agent_step_flags,
 * info) as plain host arrays, NULL members skipped; its four big members must be NULL.  This is what scales on a
 * multi-GPU node whose host memory system, not PCIe, bounds the full-format delivery (DESIGN.md 6a). */
int mapf_step_host_records(mapf_handle *h, const int8_t *actions, uint8_t *records_host, const mapf_outputs *out_host_small,
                           int32_t auto_reset);
/* The host-side ceiling of the packed path, measured: streaming fill (write-only) and copy rate, in GB/s of bytes
 * written, of the threads mapf_step_host expands with (same count, same pinning) over `bytes` of fresh memory.
 * The expansion writes every delivered byte once: delivered bytes / fill rate bounds it from below. */
int mapf_host_memory_probe(const mapf_handle *h, int64_t bytes, int32_t *threads_out, double *fill_gbs, double *copy_gbs);
/* Packed bytes per agent, and the host-side expansion on its own (no GPU needed; used by the CPU test-suite):
 * packed holds the block of n_agents agents -- [n x window+mask bits][n x (int8 d_row, int8 d_col)][n x int8
 * 2*reward] (csrc/mapf_pack_kernel.cuh); goal_delta = difference / denominator. */
int mapf_packed_record_bytes(int32_t v2);
int mapf_unpack_records(const uint8_t *packed, int64_t n_agents, int32_t v2, int32_t threads, uint8_t *local_obs,
                        int8_t *action_mask, float *goal_delta, float *reward, float den_row, float den_col);

/* ENV:306-328: pack channels into float32 flat[B,N,D] (device pointers),
 * D = V*V + 2 + gdist + bp + 5*mask, component order of ENV:214-236. */
int mapf_flat_obs_dim(const mapf_handle *h, int32_t include_goal_distance,
                      int32_t include_blocking_pressure, int32_t include_action_mask);
int mapf_pack_flat_obs(mapf_handle *h, const mapf_outputs *channels, int32_t include_goal_distance,
                       int32_t include_blocking_pressure, int32_t include_action_mask,
                       float *flat, void *stream);

/* Uniform choice among the valid actions of each agent (device int8 masks [B,N,5] ->
 * device int8 actions [B,N]); the action sampler of the reference's "masked" benchmark mode
 * (scripts/benchmark_multi_agent_env.py:42-57), Philox keyed by (seed, env id, counter). */
int mapf_sample_masked_actions(mapf_handle *h, const int8_t *action_mask, int8_t *actions,
                               uint64_t counter, void *stream);
/* Uniform actions in 0..4 (scripts/benchmark_multi_agent_env.py:38-39). */
int mapf_sample_random_actions(mapf_handle *h, int8_t *actions, uint64_t counter, void *stream);

/* Fuse the sampler into the step launch: after this call every mapf_step also writes the actions
 * for the NEXT step to next_actions (device int8 [B,N]): mode 1 = uniform over the new action
 * mask, mode 2 = uniform over 0..4, mode 0 / NULL = off.  The draw for call number c is identical
 * to mapf_sample_*_actions(..., counter = c) on the same masks; `first_counter` is the counter
 * of the next step call and increments by one per call. */
int mapf_set_fused_sampler(mapf_handle *h, int8_t *next_actions, int32_t mode, uint64_t first_counter);

/* Deterministic tree reduction of env_metrics[B,K] over the B envs into
 * device double out[MAPF_METRIC_COUNT] (off the step path; ranks then all-reduce it). */
int mapf_metrics_reduce(mapf_handle *h, double *out_device, void *stream);

/* Occupancy heat-map of the reference's evaluator (main.py:153-155, 265-267): counts[r*C+c] (device uint64 [R*C]) +=
 * the number of agents standing on (r, c), over the envs with active[env] != 0 (device uint8 [B], NULL = all). */
int mapf_occupancy_accumulate(mapf_handle *h, const uint8_t *active, uint64_t *counts, void *stream);

/* Single-agent shortest paths on the shared map (4-neighbour moves around obstacles, other agents ignored): the
 * distance field behind the reference's classical planners (scripts/a-star.py:123-126, scripts/cbs.py).
 * mapf_distance_table fills table[src * R*C + cell] (device uint8 [R*C, R*C], 255 = unreachable; maps <= 32x32);
 * mapf_goal_path_lengths writes out[b, n] = moves from agent n's position to its goal (device int16 [B,N], -1 =
 * unreachable): a lower bound of the agent's arrival time and, as the max over agents, of the makespan. */
int mapf_distance_table(mapf_handle *h, uint8_t *table, void *stream);
int mapf_goal_path_lengths(mapf_handle *h, const uint8_t *table, int16_t *out, void *stream);

/* OR of MAPF_DEV_ERR_* bits raised by kernels since the last poll (synchronises `stream`). */
int mapf_poll_errors(mapf_handle *h, uint32_t *bits, void *stream);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t mapf_launch_count(const mapf_handle *h);

/* Which step kernel this handle launches: 1 = lane-per-agent (one agent per lane, sub-warp per env),
 * 2 = env-per-thread (one env per thread, bitboards in shared memory).  Same results either way. */
int mapf_step_kernel_kind(const mapf_handle *h);

/* ------------------------------------------------------------------------------------------------
 * Single-agent ("CTE") view of the same grid world: src/environments/reference_model_single_agent.py
 * ("CTE:line") -- one joint action, one full-grid observation, one scalar reward.  Stateless entry points:
 * every buffer is a caller-owned DEVICE pointer; outputs may be NULL.
 *   ReferenceModel.step(action)   CTE:237-346 -> mapf_cte_step
 *   ReferenceModel.reset()        CTE:218-235 -> mapf_cte_reset (the caller installs positions / goals first:
 *                                                deterministic table CTE:225 or its own draw CTE:155-185)
 *   get_obs / get_action_mask     CTE:428-441, 466-489 -> obs_grid / action_mask / flat_obs outputs
 */
typedef struct mapf_cte_args {
    int32_t num_envs, num_agents, rows, cols; /* B, N <= 32, map shape */
    int32_t steps_per_episode;                /* CTE:85 */
    int32_t reserved;
    double blocking_penalty;                  /* CTE:92 */
    double move_after_goal_penalty;           /* CTE:93 */
    const uint8_t *grid;        /* [R,C] 0 free / 1 obstacle, shared by all envs */
    int16_t *positions;         /* [B,N,2] state */
    const int16_t *goals;       /* [B,N,2] */
    uint8_t *reached_once;      /* [B,N]  goal_reached_once, CTE:91 */
    int32_t *step_count;        /* [B] */
    double *blocking_total;     /* [B]    _episode_blocking_count, CTE:94 */
    const int8_t *actions;      /* [B,N]  step input (NULL = all NO_OP) */
    uint8_t *obs_grid;          /* [B,R,C] 1 obstacle, 2i+2 agent i, 2i+3 goal of agent i */
    int8_t *action_mask;        /* [B,5N] */
    float *flat_obs;            /* [B,R*C+5N] CTE:187-196 */
    double *reward;             /* [B] the Python float of the reference, bit for bit */
    uint8_t *terminated;        /* [B] */
    uint8_t *truncated;         /* [B] */
    double *info;               /* [B,4] blocking_count_step, goals_reached_step, goals_reached_total, blocking_count_total */
    uint32_t *err_bits;         /* [1] MAPF_DEV_ERR_INVALID_ACTION (required) */
    const uint8_t *reset_mask;  /* mapf_cte_reset: [B] or NULL = every env */
} mapf_cte_args;

int mapf_cte_step(const mapf_cte_args *args, void *stream);
int mapf_cte_reset(const mapf_cte_args *args, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Rollout-loop kernels around the env step (BASELINE config 5): the reference's action-mask MLP
 * (models/action_mask_model.py:8-67: Linear(F,64)-ReLU-Linear(64,64)-ReLU-{Linear(64,5), Linear(64,1)},
 * logits + log(mask + 1e-6)) evaluated straight from the env's output channels and sampled, in one launch
 * (bf16 tensor-core MLP, f32 accumulation), and generalised advantage estimation as a backwards scan.
 */
typedef struct mapf_policy_args {
    int32_t num_envs, num_agents;
    int32_t v2;           /* window cells, V * V */
    int32_t feature_dim;  /* F = v2 + 2 + (blocking_prev ? 1 : 0), <= 64: order of ENV:306-328 without the mask */
    int32_t no_masking;   /* action_mask_model.py:33 */
    int32_t greedy;       /* 0 = draw from softmax(masked logits) by inverse CDF (Philox); 1 = first index of the
                             largest masked logit (torch.argmax, RLlib forward_inference), no Philox call.  Every other
                             output is the same in both modes.  Other values: MAPF_ERR_INVALID_ARG */
    uint64_t seed;        /* Philox key (with env_id_base + env), counter = (counter, agent) */
    uint64_t counter;
    int64_t env_id_base;
    const uint8_t *local_obs;     /* [B,N,V,V]   device, the env's outputs */
    const float *goal_delta;      /* [B,N,2] */
    const uint8_t *blocking_prev; /* [B,N] or NULL */
    const int8_t *action_mask;    /* [B,N,5] */
    const void *weights;          /* device copy of the block written by mapf_policy_pack_weights */
    int8_t *actions;              /* [B,N] chosen action (feeds mapf_step), may be NULL */
    int64_t *actions64;           /* [B,N] the same as int64 (torch indexing dtype), may be NULL */
    float *logp;                  /* [B,N] log-probability of the chosen action */
    float *value;                 /* [B,N] value head */
    float *logits_out;            /* [B,N,5] masked logits, may be NULL */
    float *features_out;          /* [B,N,F] float32 feature block for the learner, may be NULL */
    int8_t *action_mask_out;      /* [B,N,5] copy of action_mask for the rollout buffer, may be NULL */
} mapf_policy_args;

/* Bytes of the packed weight block for feature_dim F (negative = unsupported F). */
int64_t mapf_policy_weights_nbytes(int32_t feature_dim);
/* HOST float32 weights in torch's Linear layout ([out, in] row-major) -> HOST packed block (bf16, padded). */
int mapf_policy_pack_weights(int32_t feature_dim, const float *w1, const float *b1, const float *w2, const float *b2,
                             const float *w_logits, const float *b_logits, const float *w_value, const float *b_value,
                             void *packed_host);
int mapf_policy_act(const mapf_policy_args *args, void *stream);

/* The recurrent policy of the reference's PPO configuration (src/agents/ppo.py:67-75): the same 64-64 ReLU trunk,
 * then an LSTM cell of 64 fed with [trunk output | one_hot(previous action, 5) | previous reward] (torch LSTMCell
 * layout, gate rows [i; f; g; o]), then logits (masked as above) and value, both reading the new h.  One launch per
 * step: features from the env's output channels, bf16 tensor-core GEMMs with f32 accumulation, the cell update in f32
 * (c stays f32), the masked inverse-CDF draw from Philox (a stream of its own, distinct from mapf_policy_act's). */
typedef struct mapf_lstm_policy_args {
    int32_t num_envs, num_agents;
    int32_t v2;           /* window cells, V * V */
    int32_t feature_dim;  /* F = v2 + 2 + (blocking_prev ? 1 : 0), <= 64: order of ENV:306-328 without the mask */
    int32_t no_masking;   /* action_mask_model.py:33 */
    int32_t greedy;       /* 0 = masked inverse-CDF draw (Philox); 1 = first index of the largest masked logit, no Philox
                             call (h_out, c_out, value, logp and logits_out as in draw mode).  Other values:
                             MAPF_ERR_INVALID_ARG */
    uint64_t seed;        /* Philox key (with env_id_base + env), counter = (counter, agent) */
    uint64_t counter;
    int64_t env_id_base;
    const uint8_t *local_obs;       /* [B,N,V,V]   device, the env's outputs */
    const float *goal_delta;        /* [B,N,2] */
    const uint8_t *blocking_prev;   /* [B,N] or NULL */
    const int8_t *action_mask;      /* [B,N,5] or NULL (no masking) */
    const uint8_t *prev_terminated; /* [B] or NULL: nonzero = this step starts an episode (h, c, previous action and */
    const uint8_t *prev_truncated;  /* [B] or NULL     previous reward count as zero for every agent of the env)     */
    const int8_t *prev_action;      /* [B,N] in 0..4, may alias `actions` (each agent's is read before it is written) */
    const float *prev_reward;       /* [B,N] */
    const float *h_in;              /* [B*N,64] LSTM state, float32 */
    const float *c_in;              /* [B*N,64] */
    float *h_out;                   /* [B*N,64] new state, may equal h_in / c_in; both NULL = do not advance the */
    float *c_out;                   /* [B*N,64]   state (h_in, c_in untouched); one NULL without the other is an error */
    const void *weights;            /* device copy of the block written by mapf_lstm_policy_pack_weights */
    int8_t *actions;                /* [B,N] chosen action (feeds mapf_step), may be NULL */
    int64_t *actions64;             /* [B,N] the same as int64, may be NULL */
    float *logp;                    /* [B,N] log-probability of the chosen action, may be NULL */
    float *value;                   /* [B,N] value head, may be NULL */
    float *logits_out;              /* [B,N,5] masked logits, may be NULL */
} mapf_lstm_policy_args;

/* Bytes of the packed LSTM policy weight block for feature_dim F (negative = unsupported F). */
int64_t mapf_lstm_policy_weights_nbytes(int32_t feature_dim);
/* HOST float32 weights in torch's layouts (Linear [out, in]; LSTMCell weight_ih [256, 70], weight_hh [256, 64],
 * b_ih / b_hh [256]) -> HOST packed block (bf16 weights, padded; b_ih + b_hh summed in f32). */
int mapf_lstm_policy_pack_weights(int32_t feature_dim, const float *w1, const float *b1, const float *w2, const float *b2,
                                  const float *w_ih, const float *w_hh, const float *b_ih, const float *b_hh,
                                  const float *w_logits, const float *b_logits, const float *w_value, const float *b_value,
                                  void *packed_host);
int mapf_lstm_policy_act(const mapf_lstm_policy_args *args, void *stream);

/* Per-agent policies (one weight set per agent, the reference's DTE mode): the same arguments, with args->weights
 * pointing to num_agents consecutive packed blocks; block j, at j * mapf_[lstm_]policy_weights_nbytes(feature_dim),
 * is written by the pack function above from agent j's parameters.  Agent j's outputs (actions, actions64, logp,
 * value, logits_out, features_out, action_mask_out; for the LSTM also h_out / c_out) equal, bit for bit, those the
 * shared entry point writes at agent j's rows when it runs with block j alone: in draw mode (the same Philox key and
 * counter) and in greedy mode, with episode-start flags, with the state updated in place or not.  The checks are
 * those of the shared entry points, plus num_agents <= MAPF_MAX_AGENTS (MAPF_ERR_UNSUPPORTED), all before any device
 * work.  A CTA works on one agent's rows at a time and reloads that agent's block into shared memory when its
 * agent changes. */
int mapf_policy_act_per_agent(const mapf_policy_args *args, void *stream);
int mapf_lstm_policy_act_per_agent(const mapf_lstm_policy_args *args, void *stream);

/* The centralised (CTE) policy over the single-agent view (cte_rollout.CteActionMaskPolicy, the restatement of
 * models/action_mask_model_single.py): the R*C grid codes of mapf_cte_step / mapf_cte_reset's obs_grid as float ->
 * Linear(R*C, 64)-ReLU-Linear(64, 64)-ReLU -> 5N logits + value, logits + log(mask + 1e-6) element by element over the
 * 5N action mask, then for every agent an independent masked 5-way draw (RLlib's multi-categorical over
 * MultiDiscrete([5] * N)), in one launch per step: bf16 tensor-core GEMMs with f32 accumulation, W1 resident in shared
 * memory.  Each agent's draw is an inverse CDF of one Philox word keyed by (seed ^ "CTEP", env_id_base + env), counter
 * (counter, agent): a stream of its own, distinct from mapf_policy_act's and mapf_lstm_policy_act's.  logp is the f32
 * sum of the agents' log-probabilities, added in agent order.
 * Supported: 1 <= num_agents <= MAPF_MAX_AGENTS and 1 <= cells <= MAPF_CTE_POLICY_MAX_CELLS (MAPF_ERR_UNSUPPORTED
 * otherwise); null inputs, num_envs < 1, reserved != 0 and greedy outside {0, 1} give MAPF_ERR_INVALID_ARG; all
 * before any device work.  greedy = 1 replaces the draws by each agent's argmax (the evaluator's mode). */
#define MAPF_CTE_POLICY_MAX_CELLS 1024

typedef struct mapf_cte_policy_args {
    int32_t num_envs, num_agents;
    int32_t cells;                 /* R * C */
    int32_t reserved;              /* must be 0 */
    uint64_t seed;
    uint64_t counter;
    int64_t env_id_base;
    const uint8_t *obs_grid;       /* [B, cells] device, the CTE env's grid codes */
    const int8_t *action_mask;     /* [B, 5N] */
    const void *weights;           /* device copy of the block written by mapf_cte_policy_pack_weights */
    int8_t *actions;               /* [B, N] joint action (feeds mapf_cte_step), may be NULL */
    int64_t *actions64;            /* [B, N] the same as int64, may be NULL */
    float *logp;                   /* [B] joint log-probability, may be NULL */
    float *value;                  /* [B] value head, may be NULL */
    float *logits_out;             /* [B, N, 5] masked logits, may be NULL */
    int32_t greedy;                /* 0 = the per-agent draws above; 1 = per agent the first index of the largest masked
                                      logit (torch.argmax, RLlib's deterministic MultiDiscrete sample), no Philox call, so
                                      seed and counter do not matter; logp is then the sum of the chosen actions'
                                      log-probabilities, every other output is what draw mode writes.  Other values:
                                      MAPF_ERR_INVALID_ARG */
} mapf_cte_policy_args;

/* Bytes of the packed CTE policy weight block (negative = unsupported cells / num_agents). */
int64_t mapf_cte_policy_weights_nbytes(int32_t cells, int32_t num_agents);
/* HOST float32 weights in torch's Linear layout (w1 [64, cells], w2 [64, 64], w_logits [5N, 64], w_value [1, 64]) ->
 * HOST packed block (bf16 weights, padded; f32 biases). */
int mapf_cte_policy_pack_weights(int32_t cells, int32_t num_agents, const float *w1, const float *b1, const float *w2,
                                 const float *b2, const float *w_logits, const float *b_logits, const float *w_value,
                                 const float *b_value, void *packed_host);
int mapf_cte_policy_act(const mapf_cte_policy_args *args, void *stream);

/* The recurrent centralised (CTE) policy (cte_rollout.CteRecurrentPolicy, the reference's PPO model of
 * src/agents/ppo.py:67-75 on the single-agent view): the grid codes -> the 64-64 ReLU trunk of mapf_cte_policy_act ->
 * an LSTM cell of 64 fed with [trunk output | one-hot of the previous joint action (the N five-way one-hots in agent
 * order) | previous reward] (torch LSTMCell layout, gate rows [i; f; g; o]) -> 5N logits (masked as above) and the
 * value, both reading the new h -> the N masked draws.  Two launches per call on `stream`: the trunk (bf16 output
 * into the caller's `trunk` workspace), then the recurrent step (bf16 gate GEMM with f32 accumulation, the reward
 * term added in f32, c kept in f32) with the heads and the draws.  Each agent's draw is an inverse CDF of one Philox
 * word keyed by (seed ^ "CTEL", env_id_base + env), counter (counter, agent): a stream of its own; logp is the f32 sum
 * of the agents' log-probabilities in agent order.  Supported shapes are mapf_cte_policy_act's
 * (MAPF_ERR_UNSUPPORTED otherwise); null required pointers, num_envs < 1, reserved != 0, greedy outside {0, 1} and
 * h_out without c_out (or the reverse) give MAPF_ERR_INVALID_ARG; all before any device work. */
typedef struct mapf_cte_lstm_policy_args {
    int32_t num_envs, num_agents;
    int32_t cells;                  /* R * C */
    int32_t reserved;               /* must be 0 */
    uint64_t seed;
    uint64_t counter;
    int64_t env_id_base;
    const uint8_t *obs_grid;        /* [B, cells] device, the CTE env's grid codes */
    const int8_t *action_mask;      /* [B, 5N] */
    const uint8_t *prev_terminated; /* [B] or NULL: nonzero = this step starts an episode (h, c, previous action and */
    const uint8_t *prev_truncated;  /* [B] or NULL     previous reward count as zero)                                */
    const int8_t *prev_action;      /* [B, N] in 0..4, may alias `actions` (an env's are read before they are written) */
    const double *prev_reward;      /* [B] the CTE env's own reward type */
    const float *h_in;              /* [B, 64] LSTM state, float32 */
    const float *c_in;              /* [B, 64] */
    float *h_out;                   /* [B, 64] new state, may equal h_in / c_in; both NULL = do not advance the state */
    float *c_out;                   /* [B, 64]   (h_in, c_in untouched); one NULL without the other is an error */
    void *trunk;                    /* [B, 64] bf16 workspace: the trunk output, written by the first launch */
    const void *weights;            /* device copy of the block written by mapf_cte_lstm_policy_pack_weights */
    int8_t *actions;                /* [B, N] joint action (feeds mapf_cte_step), may be NULL */
    int64_t *actions64;             /* [B, N] the same as int64, may be NULL */
    float *logp;                    /* [B] joint log-probability, may be NULL */
    float *value;                   /* [B] value head, may be NULL */
    float *logits_out;              /* [B, N, 5] masked logits, may be NULL */
    int32_t greedy;                 /* 0 = draw; 1 = per agent the first argmax of the masked logits, no Philox call
                                       (h_out, c_out, trunk, value, logp and logits_out as in draw mode); other values:
                                       MAPF_ERR_INVALID_ARG.  As mapf_cte_policy_args.greedy */
} mapf_cte_lstm_policy_args;

/* Bytes of the packed recurrent CTE policy weight block (negative = unsupported cells / num_agents). */
int64_t mapf_cte_lstm_policy_weights_nbytes(int32_t cells, int32_t num_agents);
/* HOST float32 weights in torch's layouts (Linear [out, in]: w1 [64, cells], w2 [64, 64], w_logits [5N, 64],
 * w_value [1, 64]; LSTMCell weight_ih [256, 64 + 5N + 1], weight_hh [256, 64], b_ih / b_hh [256]) -> HOST packed
 * block (bf16 weights, padded; the reward column of weight_ih and the biases in f32, b_ih + b_hh summed in f32). */
int mapf_cte_lstm_policy_pack_weights(int32_t cells, int32_t num_agents, const float *w1, const float *b1,
                                      const float *w2, const float *b2, const float *w_ih, const float *w_hh,
                                      const float *b_ih, const float *b_hh, const float *w_logits,
                                      const float *b_logits, const float *w_value, const float *b_value,
                                      void *packed_host);
int mapf_cte_lstm_policy_act(const mapf_cte_lstm_policy_args *args, void *stream);
/* Per-step bookkeeping of the batched evaluator (main.py:test_trained_model, one episode per env, no auto-reset), in
 * one launch after mapf_step (and after mapf_occupancy_accumulate, which reads `active` before this call clears it).
 * For every env with active[b] != 0: episode_reward[b] += sum of the agents' rewards (main.py:251), agent_reward[b,n]
 * += reward[b,n] (main.py:262), timesteps[b] += 1, last_info[b,:] = info[b,:]; if terminated[b] | truncated[b] the
 * episode ends: success[b] = terminated[b] && !truncated[b] (main.py:294) and active[b] = 0.  Inactive envs are not
 * touched.  The envs still active after the call are counted into active_count[step & 1], which must be zero on entry;
 * the call zeroes active_count[(step & 1) ^ 1] for the next call, so a loop that passes step = 0, 1, 2, ... starting
 * from two zero words needs no memset between steps and reads one word per step.  Every pointer is a device pointer
 * and is required. */
typedef struct mapf_eval_args {
    int32_t num_envs, num_agents;
    int64_t step;               /* selects the counter word, see above */
    const float *reward;        /* [B,N] this step's rewards */
    const uint8_t *terminated;  /* [B] */
    const uint8_t *truncated;   /* [B] */
    const int32_t *info;        /* [B,16] */
    uint8_t *active;            /* [B] 1 while the env's first episode runs; cleared by this call at its end */
    double *episode_reward;     /* [B] */
    double *agent_reward;       /* [B,N] */
    int64_t *timesteps;         /* [B] */
    uint8_t *success;           /* [B] */
    int32_t *last_info;         /* [B,16] info of the env's last active step */
    uint32_t *active_count;     /* [2] envs still active after this step, in word step & 1 */
} mapf_eval_args;

int mapf_eval_accumulate(const mapf_eval_args *args, void *stream);

/* The same bookkeeping for the single-agent (CTE) view (mapf_cte_step's outputs: one f64 reward per env, f64 [B,4]
 * info, int16 [B,N,2] positions), stateless, one call per step after mapf_cte_step.  It first adds the heat-map:
 * occupancy[r * cols + c] += 1 for every agent of every env with active[b] != 0 at its position (r, c) after the step
 * (main.py:264-267, positions outside the map are skipped).  Then, for every env with active[b] != 0:
 * episode_reward[b] += reward[b] (in step order, bit for bit a Python `total += reward` loop), timesteps[b] += 1,
 * last_info[b,:] = info[b,:]; if terminated[b] | truncated[b]: success[b] = terminated[b] && !truncated[b] and
 * active[b] = 0.  active_count follows mapf_eval_accumulate's parity scheme (word step & 1 counts the envs still
 * active, the other word is zeroed).  Every pointer is a device pointer and is required; null pointers or a
 * non-positive num_envs / num_agents / rows / cols give MAPF_ERR_INVALID_ARG, num_agents > MAPF_MAX_AGENTS
 * MAPF_ERR_UNSUPPORTED, all before any device work. */
#define MAPF_CTE_INFO_WORDS 4

typedef struct mapf_cte_eval_args {
    int32_t num_envs, num_agents, rows, cols;
    int64_t step;               /* selects the counter word */
    const int16_t *positions;   /* [B,N,2] (row, col) after the step */
    const double *reward;       /* [B] */
    const uint8_t *terminated;  /* [B] */
    const uint8_t *truncated;   /* [B] */
    const double *info;         /* [B,4] as mapf_cte_args.info */
    uint8_t *active;            /* [B] 1 while the env's first episode runs; cleared by this call at its end */
    double *episode_reward;     /* [B] */
    int64_t *timesteps;         /* [B] */
    uint8_t *success;           /* [B] */
    double *last_info;          /* [B,4] info of the env's last active step */
    uint64_t *occupancy;        /* [rows * cols] */
    uint32_t *active_count;     /* [2] envs still active after this step, in word step & 1 */
} mapf_cte_eval_args;

int mapf_cte_eval_accumulate(const mapf_cte_eval_args *args, void *stream);

/* rewards / values / adv / ret: device float32 [T,B,N]; dones uint8 [T,B]; last_value float32 [B,N]. */
int mapf_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_value, float *adv,
             float *ret, int32_t T, int64_t B, int32_t N, float gamma, float lam, void *stream);

/* V-trace targets (IMPALA, Espeholt et al. 2018; RLlib's vtrace_torch recurrence with c_bar fixed at 1) over M time
 * columns of a rollout, one thread per column, a backwards scan in f32.  A batch column is one (env, agent) series,
 * col = env * num_agents + agent (num_agents = 1 for the CTE view).  Processed column m reads batch column
 * col = columns[m] (columns == NULL: col = m, M = num_columns).  For t = T-1 .. 0, with mu / pi the behaviour / target
 * log-probabilities, V the values, r the rewards, d the episode ends (terminated or truncated) and V_T the bootstrap:
 *   rho_t = exp(pi_t - mu_t); rho_bar_t = min(clip_rho, rho_t); c_t = min(1, rho_t); rho_pg_t = min(clip_pg_rho, rho_t)
 *   disc_t = gamma * (1 - d_t); delta_t = rho_bar_t * (r_t + disc_t * V_{t+1} - V_t)      (V_{t+1} = V_T at t = T-1)
 *   acc_T = 0; acc_t = delta_t + disc_t * c_t * acc_{t+1}; vs_t = V_t + acc_t
 *   pg_adv_t = rho_pg_t * (r_t + disc_t * vs_{t+1} - V_t)                                  (vs_T = V_T)
 * Every pointer is a device pointer; all are required except `columns`.  Null required pointers, T < 1, M < 1,
 * num_agents < 1, num_columns not a positive multiple of num_agents, columns == NULL with M != num_columns, gamma
 * outside [0, 1], a non-finite or non-positive clip threshold and reserved != 0 give MAPF_ERR_INVALID_ARG, all before
 * any device work.  On the device, a column id outside [0, num_columns) writes NaN to that column's outputs and reads
 * no input. */
typedef struct mapf_vtrace_args {
    int32_t T, num_agents;          /* time steps; columns per env (1 for the CTE view) */
    int64_t num_columns, M;         /* batch columns (B * num_agents); processed columns */
    const int64_t *columns;         /* [M] batch column ids, or NULL for 0 .. M-1 */
    const float *rewards;           /* [T, num_columns] */
    const float *behaviour_logp;    /* [T, num_columns] */
    const uint8_t *dones;           /* [T, num_columns / num_agents], 0 / nonzero (torch bool bytes as they are) */
    const float *bootstrap_value;   /* [num_columns] value of the observation after step T-1 */
    const float *target_logp;       /* [T, M] */
    const float *values;            /* [T, M] */
    float *vs;                      /* [T, M] out */
    float *pg_advantages;           /* [T, M] out */
    float gamma, clip_rho, clip_pg_rho;
    int32_t reserved;               /* must be 0 */
} mapf_vtrace_args;

int mapf_vtrace(const mapf_vtrace_args *args, void *stream);

/* ------------------------------------------------------------------------------------------------
 * DQN (the reference's src/agents/dqn.py, SURVEY §2 row 6): an epsilon-greedy dueling Q kernel over the fused MLP's
 * packed weights, and a prioritized replay sum tree on the device.
 *
 * mapf_q_act / mapf_q_act_per_agent: the MLP of mapf_policy_act (the same packed block, per agent: num_agents blocks)
 * read as a dueling network: logits head = advantage A[5], value head = V, Q = V + (A - mean(A)) in f32 with the mean
 * over all 5 actions; masked Q = Q where the mask allows the action, FLOAT_MIN (-3.4e38) elsewhere (no_masking: Q as it
 * is).  Per agent, with one Philox block keyed (seed ^ "DQNE", env_id_base + env), counter (counter, agent): explore
 * iff word0 * 2^-32 < epsilon, then take the k-th legal action (all 5 with no_masking), k = floor(word1 * n_legal /
 * 2^32); otherwise the first index of the largest masked Q (torch.argmax's tie rule).  epsilon = 0 makes no Philox
 * call.  Null required pointers (local_obs, goal_delta, action_mask, weights, actions), num_envs or num_agents < 1,
 * epsilon outside [0, 1] or NaN and reserved != 0 give MAPF_ERR_INVALID_ARG; a feature_dim that does not match v2 (as
 * in mapf_policy_act), and for the per-agent entry num_agents > MAPF_MAX_AGENTS, give MAPF_ERR_UNSUPPORTED; all
 * before any device work. */
typedef struct mapf_q_act_args {
    int32_t num_envs, num_agents;
    int32_t v2;           /* window cells, V * V */
    int32_t feature_dim;  /* F = v2 + 2 + (blocking_prev ? 1 : 0), <= 64 */
    int32_t no_masking;   /* action_mask_model.py:33: nonzero = Q unmasked, explore over all 5 actions */
    float epsilon;        /* exploration probability in [0, 1] */
    uint64_t seed;        /* Philox key (with env_id_base + env), counter = (counter, agent) */
    uint64_t counter;
    int64_t env_id_base;
    const uint8_t *local_obs;     /* [B,N,V,V]   device, the env's outputs */
    const float *goal_delta;      /* [B,N,2] */
    const uint8_t *blocking_prev; /* [B,N] or NULL */
    const int8_t *action_mask;    /* [B,N,5] */
    const void *weights;          /* device copy of the block(s) written by mapf_policy_pack_weights */
    int8_t *actions;              /* [B,N] chosen action */
    float *q_out;                 /* [B,N,5] masked Q, may be NULL */
    int32_t reserved;             /* must be 0 */
} mapf_q_act_args;

int mapf_q_act(const mapf_q_act_args *args, void *stream);
int mapf_q_act_per_agent(const mapf_q_act_args *args, void *stream);

/* Prioritized replay over a ring of `capacity` env steps (K slots) of num_envs (B) envs x num_agents (N) agents.
 * Transition (slot k, env b, agent j) has the flat index (k * B + b) * N + j.  The tree is an implicit binary heap
 * over L = N' K' B' leaves (N', K', B' = N, K, B rounded up to powers of two), leaves ordered (agent, slot, env): leaf
 * (j K' + k) B' + b.  Arrays (device, allocated by the caller):
 *   leaves [L] float32: p^alpha of a complete transition, 0 for a slot without one (never drawn) and for padding;
 *   sums   [L] float64: node i in 1 .. L-1 holds the sum of its children 2i, 2i+1 (node L + l is leaf l);
 *   mins   [L] float32: the minimum over the nonzero leaves below node i, +inf when there are none;
 *   max_priority [1] float32: the largest priority (not raised to alpha) seen so far, 1.0 for a new buffer.
 * A fresh tree is leaves 0, sums 0, mins +inf.  Agent j's transitions form the subtree of node N' + j.
 * Every entry point refuses null pointers, num_envs, num_agents or M < 1, capacity < 2, a negative or non-finite
 * alpha / beta and reserved != 0 with MAPF_ERR_INVALID_ARG, before any device work. */
int64_t mapf_replay_tree_leaves(int32_t num_envs, int32_t num_agents, int32_t capacity);   /* L, or a MAPF_ERR_* */

typedef struct mapf_replay_tree {
    int32_t num_envs, num_agents, capacity;
    float *leaves;
    double *sums;
    float *mins;
    float *max_priority;
} mapf_replay_tree;

/* One env step of the ring: every (b, j) leaf of slot `complete` becomes max_priority^alpha, every leaf of slot `clear`
 * becomes 0, then the nodes above them are recomputed.  Deterministic: every node is the sum (minimum) of its two
 * children, with no float atomics.  complete and clear must differ and lie in [0, capacity) (MAPF_ERR_INVALID_ARG). */
typedef struct mapf_replay_advance_args {
    mapf_replay_tree tree;
    int32_t complete, clear;
    float alpha;
    int32_t reserved;             /* must be 0 */
} mapf_replay_advance_args;

/* M i.i.d. proportional draws (RLlib's _sample_proportional): u in [0, 1) from one Philox block keyed (seed ^ "PRPS",
 * draw), counter (counter); target = u * total; descend from the root to the first leaf whose prefix sum exceeds the
 * target.  per_agent: draw i descends from agent (i mod N)'s subtree, with that agent's total and minimum.  Writes
 * the transition's flat index and the importance weight w = (P(i) n)^-beta / ((p_min / total) n)^-beta
 * = (p_i / p_min)^-beta, computed in f64 (n cancels); `uniforms` (optional) receives u.  An empty (sub)tree writes
 * index -1 and weight 0. */
typedef struct mapf_replay_sample_args {
    mapf_replay_tree tree;
    int64_t M;
    uint64_t seed, counter;
    float beta;
    int32_t per_agent;
    int64_t *indices;             /* [M] out */
    float *weights;               /* [M] out */
    double *uniforms;             /* [M] out, may be NULL */
    int32_t reserved;             /* must be 0 */
} mapf_replay_sample_args;

/* New priorities for M transitions: leaf = (|delta| + 1e-6)^alpha for every in-range index whose leaf is nonzero
 * (out-of-range indices and transitions of cleared slots are skipped; among duplicates the largest value is kept, so
 * the result does not depend on thread order), max_priority = max(max_priority, |delta| + 1e-6) over those, then the
 * ancestors are recomputed level by level.  One block. */
typedef struct mapf_replay_update_args {
    mapf_replay_tree tree;
    int64_t M;
    const int64_t *indices;       /* [M] flat transition indices */
    const float *td_abs;          /* [M] |TD error| */
    float alpha;
    int32_t reserved;             /* must be 0 */
} mapf_replay_update_args;

int mapf_replay_advance(const mapf_replay_advance_args *args, void *stream);
int mapf_replay_sample(const mapf_replay_sample_args *args, void *stream);
int mapf_replay_update(const mapf_replay_update_args *args, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Prioritized planner on the handle's shared map (maps <= 32x32, the classical-planner baseline of scripts/a-star.py
 * and scripts/cbs.py under this env's own move rule).  Agents plan in index order; agent i finds its earliest arrival
 * by a space-time wavefront that avoids the cells the agents before it hold, under the rule of mapf_step (ENV:502-526:
 * a move into a cell held by a lower index at its new position or by a higher index at its old position fails), with
 * the unplanned agents on their starts at t = 0 and every planned agent on its goal from its arrival on.  Among paths
 * with the same arrival it takes, walking back from the goal, the first predecessor in the action order NO_OP, UP,
 * RIGHT, DOWN, LEFT; there is no RNG, so the same layouts give the same plan.  An agent with no arrival within the
 * horizon, an unreachable goal, or a start / goal off the map gets arrival -1 and NO_OP actions, and (on the map)
 * reserves its start for every t; the other agents are still planned.  status[b] = 1 iff every agent of env b
 * arrived; only then do the actions replay through mapf_step without a failed move and end the episode (terminated)
 * at step max(1, max arrival) with every agent on its goal.  DESIGN.md §7 N4b.
 *
 * Refused before any device work: a null handle, args or buffer, num_envs < 1, num_agents < 1, horizon < 1,
 * reserved != 0 or a workspace smaller than mapf_plan_workspace_bytes give MAPF_ERR_INVALID_ARG; num_agents >
 * MAPF_MAX_AGENTS, per-env maps and maps wider or taller than 32 give MAPF_ERR_UNSUPPORTED; a handle without a map
 * MAPF_ERR_STATE. */
typedef struct mapf_plan_args {
    int32_t num_envs, num_agents;   /* B (independent of the handle's num_envs), N */
    int32_t horizon;                /* H: steps a plan may take (the env's steps_per_episode) */
    int32_t reserved;               /* must be 0 */
    const int16_t *starts;          /* [B,N,2] (row, col) device */
    const int16_t *goals;           /* [B,N,2] */
    const uint8_t *distance_table;  /* [R*C, R*C] written by mapf_distance_table for this handle */
    void *workspace;                /* device scratch of workspace_bytes, contents need not be initialised */
    int64_t workspace_bytes;
    int8_t *actions;                /* [H,B,N] out: action of agent n of env b at step t */
    int16_t *arrival;               /* [B,N] out: arrival step, 0 for an agent that starts on its goal, -1 = none */
    uint8_t *status;                /* [B] out: 1 = every agent arrived */
} mapf_plan_args;

/* Workspace bytes of mapf_plan_prioritized for a rows x cols map, num_envs envs and horizon H, or a MAPF_ERR_* code
 * (MAPF_ERR_INVALID_ARG for non-positive arguments, MAPF_ERR_UNSUPPORTED for maps over 32x32). */
int64_t mapf_plan_workspace_bytes(int32_t rows, int32_t cols, int32_t num_envs, int32_t horizon);
int mapf_plan_prioritized(mapf_handle *h, const mapf_plan_args *args, void *stream);

/* Windowed prioritized planner for rolling-horizon replanning (RHCR, Li et al. 2021) from any state, lifelong envs
 * included: the rule of mapf_plan_prioritized with the horizon read as the window W (args->horizon; actions [W,B,N]),
 * resolving conflicts only within W and not requiring arrival.  The target is the goal if distance_table reaches it
 * from the start (!= 255), else the start.  An agent with the goal as target arrives at the first t <= W with the
 * goal in its wavefront and t >= max(d, last hold of the goal + 1), and holds it to W (arrival = t).  Otherwise the
 * search runs to t = W and the path ends on the cell of the wavefront at W with the smallest distance-table value
 * from the target, ties to the first cell in row-major order; the agent reserves that path and gets arrival -1.  An
 * agent whose wavefront empties before W, or whose start or goal lies off the map, fails as in mapf_plan_prioritized
 * (NO_OPs, start reserved for every t); the later agents are still planned.  status[b] = 1 iff every agent of env b
 * got a path; then replaying the W actions through mapf_step from the planned state gives no failed move and every
 * agent follows its planned cells (also in lifelong mode: goal reassignment never moves an agent), and an agent that
 * arrived stands on its goal from its arrival on.  On envs where mapf_plan_prioritized at H gives status 1, the
 * windowed plan at W = H has the same actions and arrivals.  Refusals are those of mapf_plan_prioritized, before any
 * device work; mapf_plan_workspace_bytes(rows, cols, B, W) sizes the workspace.  DESIGN.md §7 N4c. */
int mapf_plan_windowed(mapf_handle *h, const mapf_plan_args *args, void *stream);

/* Conflict-based search (CBS) on the handle's shared map under mapf_step's move rule: per env, a plan with the least
 * sum of arrivals within the horizon, or the reason there is none.  A joint plan (every agent on its goal from its
 * arrival on) replays without a failed move iff no two agents share a cell at t + 1 (vertex) and no agent a moves at t
 * into the cell a higher index b holds at t (following); each conflict splits into two vertex constraints, (a, c, t+1)
 * / (b, c, t+1) and (a, c, t+1) / (b, c, t).  The low level is the wavefront of mapf_plan_prioritized with the agent's
 * constraints as the only obstacles besides the map: earliest arrival t <= H with t > every constrained t of the goal,
 * the same backtrack tie rule.  The high level pops the open node of least (sum of arrivals, creation id), takes its
 * first conflict (smallest t; vertex before following; lowest a, then lowest b) and creates the child constraining a,
 * then the one constraining b, replanning only that agent; a child without a path is not created.  Deterministic: the
 * same layouts give the same plan and expansion count.  DESIGN.md §7 N4d.
 *
 * status[b] (the outcome): 1 = the popped node has no conflict: an optimal plan, whose actions replay through mapf_step
 * without a failed move and end the episode (terminated) at step max(1, max arrival) with every agent on its goal;
 * 0 = no plan exists within the horizon (an agent with no path, a start or goal off the map, on an obstacle or repeated
 * -- these without a search, expanded = 0 -- or the open list exhausted); 2 = max_nodes expansions without an answer.
 * Outcomes 0 and 2 give NO_OP actions and arrival -1.  expanded[b] = the nodes popped.
 *
 * Refused before any device work: those of mapf_plan_prioritized (with mapf_cbs_workspace_bytes for the size), and
 * max_nodes outside 1..65536 or horizon > 32767 (MAPF_ERR_INVALID_ARG).  The launch first zeroes the workspace's env
 * counter with cudaMemsetAsync on `stream`; envs are taken from it by one warp each.  CBS is for small agent counts
 * (2-8): its search grows with the number of conflicts; mapf_plan_prioritized stays the large-N baseline. */
typedef struct mapf_cbs_args {
    int32_t num_envs, num_agents;   /* B, N */
    int32_t horizon;                /* H */
    int32_t max_nodes;              /* K: the expansion budget, 1..65536 */
    const int16_t *starts;          /* [B,N,2] (row, col) device */
    const int16_t *goals;           /* [B,N,2] */
    const uint8_t *distance_table;  /* [R*C, R*C] written by mapf_distance_table for this handle */
    void *workspace;                /* device scratch of workspace_bytes, contents need not be initialised */
    int64_t workspace_bytes;
    int8_t *actions;                /* [H,B,N] out */
    int16_t *arrival;               /* [B,N] out: arrival step for outcome 1, else -1 */
    uint8_t *status;                /* [B] out: the outcome 0 / 1 / 2 */
    int32_t *expanded;              /* [B] out: high-level nodes popped */
    int32_t reserved;               /* must be 0 */
} mapf_cbs_args;

/* Workspace bytes of mapf_plan_cbs, or a MAPF_ERR_* code (MAPF_ERR_INVALID_ARG for non-positive arguments, max_nodes
 * over 65536 or horizon over 32767, MAPF_ERR_UNSUPPORTED for maps over 32x32 or num_agents over MAPF_MAX_AGENTS):
 *   16 + num_envs * ceil16(24 (2K + 1) + 64 + 8 (H + 1) rows + (N + 2K) ceil16(H))
 * (a 16-byte env counter; per env the node records and open-list keys, the root's arrivals, the constraint and
 * wavefront planes, and one int8 action path per root agent and per child).  65 536 envs at N = 8, H = 256, K = 1024
 * take 42 GB; the path slots dominate, so size K to the search the layouts need. */
int64_t mapf_cbs_workspace_bytes(int32_t rows, int32_t cols, int32_t num_envs, int32_t num_agents, int32_t horizon,
                                 int32_t max_nodes);
int mapf_plan_cbs(mapf_handle *h, const mapf_cbs_args *args, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MAPF_B200_H */
