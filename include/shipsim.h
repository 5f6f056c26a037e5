/*
 * shipsim.h -- C ABI of libshipsim.so, the B200-native batched replacement for the CapAI/ship-sim-gym
 * environment step.
 *
 * The reference has no FFI of its own for this path: the boundary it exposes is the gym `Env` protocol of
 * `ShipEnv` (ship_gym/ship_env.py:16-184), and everything below that line is Python + pymunk.  This header is
 * what a maintainer's ctypes stub inside ShipEnv would bind (INTEGRATION.md shows that stub); each entry point
 * cites the reference interface it replaces (file:line under the reference tree).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types.  `stream` is a cudaStream_t passed as void*
 *     (NULL = legacy default stream).
 *   - every function returns 0 on success or a negative shipsim_status; the message of the last failure on the
 *     calling thread is available from shipsim_last_error().  Nothing throws across the ABI.
 *   - pointers named dev_* are device pointers valid on the handle's device and owned by the CALLER (in the
 *     Python host layer they are torch tensors); pointers named host_* are host memory.
 *   - shipsim_step / shipsim_reset / shipsim_stats_read allocate nothing and never synchronise: all work is
 *     enqueued on the caller's stream, so they are CUDA-graph capturable.
 *   - a handle is not thread-safe; use one handle per GPU per process (one process per GPU when sharding).
 *   - there is no CPU fallback: every call fails with SHIPSIM_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef SHIPSIM_H
#define SHIPSIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHIPSIM_ABI_VERSION 4
#define SHIPSIM_N_GOALS 5        /* game.py:17  N_GOALS */
#define SHIPSIM_N_BEAMS 10       /* models.py:29 LiDAR(n_beams=10): the only beam count the reference ever uses; the default */
#define SHIPSIM_MAX_BEAMS 32     /* widest lidar fan (lidar_beams in [1, SHIPSIM_MAX_BEAMS])                               */
#define SHIPSIM_FRAME 16         /* ship_env.py:43 n_states = 2+1+1+2+n_beams */
#define SHIPSIM_STATE_PLANES 8   /* float4 planes per env, see shipsim_state_bytes() */
#define SHIPSIM_MAX_HULL 32      /* max convex-hull vertices per river bank */
#define SHIPSIM_STATS_LEN 16

typedef enum shipsim_status {
    SHIPSIM_OK = 0,
    SHIPSIM_ERR_ARG = -1,        /* bad argument (ValueError on the Python side) */
    SHIPSIM_ERR_CUDA = -2,       /* CUDA runtime failure / no usable device */
    SHIPSIM_ERR_STATE = -3,      /* call order: state or scenarios not bound yet */
    SHIPSIM_ERR_UNSUPPORTED = -4
} shipsim_status;

typedef enum shipsim_action_dtype {
    SHIPSIM_ACTION_I32 = 0,
    SHIPSIM_ACTION_I64 = 1,      /* what torch.multinomial / argmax produce: no cast kernel needed */
    SHIPSIM_ACTION_U8 = 2,
    SHIPSIM_ACTION_RANDOM = 3    /* dev_actions ignored: uniform{0,1,2} from Philox(seed, env, step) -- the
                                    random agent of train/random.py:18 */
} shipsim_action_dtype;

/* Episode statistics, one double each (so the 128-byte vector can go straight into an all-reduce(SUM)). */
typedef enum shipsim_stat {
    SHIPSIM_STAT_EPISODES = 0,   /* finished episodes                                   */
    SHIPSIM_STAT_RETURN_SUM,     /* sum of ShipEnv.cumulative_reward at episode end (ship_env.py:150) */
    SHIPSIM_STAT_LENGTH_SUM,     /* sum of ShipEnv.step_count at episode end (ship_env.py:152)        */
    SHIPSIM_STAT_GOAL_STEPS,     /* steps on which game.goal_reached was set (game.py:254)            */
    SHIPSIM_STAT_COLLISION,      /* episodes that ended with game.colliding (ship_env.py:120)         */
    SHIPSIM_STAT_OOB,            /* ... out of bounds (ship_env.py:126-129)                           */
    SHIPSIM_STAT_TIMEOUT,        /* ... step_count >= MAX_STEPS (ship_env.py:131)                     */
    SHIPSIM_STAT_ALL_GOALS,      /* ... no goals left (ship_env.py:122)                               */
    SHIPSIM_STAT_STEPS           /* env-steps executed                                                 */
} shipsim_stat;

/* Episode log (shipsim_episode_log_bind): one record per finished episode, 8 int32 of metadata + the terminal row. */
#define SHIPSIM_EPISODE_META 8
enum {
    SHIPSIM_EP_K = 0,            /* step index within the caller's shipsim_step / shipsim_step_host call   */
    SHIPSIM_EP_ENV,              /* local env index                                                          */
    SHIPSIM_EP_LENGTH,           /* ShipEnv.step_count at episode end (ship_env.py:152)                      */
    SHIPSIM_EP_RETURN,           /* ShipEnv.cumulative_reward at episode end (ship_env.py:150), float bits   */
    SHIPSIM_EP_END,              /* why it ended: SHIPSIM_END_* bits, possibly several                       */
    SHIPSIM_EP_SCENARIO,         /* the finished episode's scenario ...                                      */
    SHIPSIM_EP_EPISODE,          /* ... and episode number                                                   */
    SHIPSIM_EP_CALL              /* the handle's sequence number of the step call, taken at enqueue         */
};
/* Per-map level scores (shipsim_gae_scored): one row of doubles per scenario, then one row for steps of no known scenario. */
enum {
    SHIPSIM_SCORE_STEPS = 0,     /* rollout steps played on the map                                          */
    SHIPSIM_SCORE_POS_ADV,       /* sum over those steps of max(GAE advantage, 0): PLR's positive value loss  */
    SHIPSIM_SCORE_ABS_ADV,       /* sum over those steps of |GAE advantage|: the L1 value loss                */
    SHIPSIM_SCORE_COLS
};
enum {
    SHIPSIM_END_COLLISION = 1,   /* game.colliding (ship_env.py:120)          */
    SHIPSIM_END_ALL_GOALS = 2,   /* no goals left (ship_env.py:122)           */
    SHIPSIM_END_OOB = 4,         /* out of bounds (ship_env.py:126-129)       */
    SHIPSIM_END_TIMEOUT = 8,     /* step_count >= MAX_STEPS (ship_env.py:131): the only truncation */
    SHIPSIM_END_GOAL = 16        /* a goal was taken on the last step         */
};

/* Knobs.  Mirrors ship_gym/config.py:14-24 (GameConfig / EnvConfig) plus the constants the reference
 * hard-codes; the host layer fills it from those classes.  Zero-initialise, then call
 * shipsim_config_default(). */
typedef struct shipsim_config {
    int32_t struct_size;         /* = sizeof(shipsim_config), checked by shipsim_create              */
    int32_t num_envs;            /* envs owned by this handle (this rank's shard)                    */
    int64_t env_id_offset;       /* global id of local env 0: RNG streams are keyed by global id so
                                    results do not depend on how envs are sharded over GPUs          */
    uint64_t seed;
    float bounds_w, bounds_h;    /* GameConfig.BOUNDS            config.py:24                         */
    float dt;                    /* GameConfig.SPEED * base_dt   config.py:23, game.py:27,194         */
    float damping;               /* pow(space.damping=0.4, dt)   game.py:270 -- computed in double by the host */
    int32_t max_steps;           /* EnvConfig.MAX_STEPS          config.py:16                         */
    int32_t history;             /* EnvConfig.HISTORY_SIZE       config.py:15 ; 1 or 2 here, the host layer
                                    builds longer histories from the frames                           */
    int32_t auto_reset;          /* 1: a done env is reset inside the step and its obs replaced by the reset
                                    obs (the SubprocVecEnv worker behind train/stable_baselines/ppo.py:123) */
    int32_t lidar_beams;         /* rays of the fan, 1..32 (LidarConfig.N_BEAMS config.py:9 when honoured; default
                                    SHIPSIM_N_BEAMS).  An observation frame is 6 + lidar_beams floats.  10 runs the tuned
                                    kernels; any other count the wide serial-in-time kernel: steps_in_flight must then be
                                    0 or 1 (SHIPSIM_ERR_UNSUPPORTED otherwise)                       */
    float lidar_spread_deg;      /* models.py:29 (90); LidarConfig.ANGULAR_SPREAD config.py:11 when honoured */
    float lidar_distance;        /* models.py:29 (100)                                               */
    float ship_w, ship_h;        /* game.py:275 (2, 3): scale of models.py:6 SHIP_TEMPLATE           */
    float mass;                  /* models.py:87 (5)                                                 */
    float thrust;                /* models.py:107 (100)                                              */
    float goal_radius;           /* game.py:82 (5)                                                   */
    float step_penalty;          /* ship_env.py:13 (-0.01)                                           */
    float spawn_y;               /* game.py:274 (25); spawn x is bounds_w/2                          */
    int32_t lanes_per_env;       /* cooperating lanes per env: 0 = choose from num_envs, else 1, 2, 4, 8, 16 or 32
                                    (32 = one warp per env, for small latency-bound batches)         */
    int32_t steps_in_flight;     /* K-step rollouts of small batches: consecutive steps of one env speculated together
                                    (the rigid-body recurrence is cheap and sequential; lidar, overlap and goal tests
                                    of different steps run on different lanes; the window is cut at the first `done`).
                                    0 = choose from num_envs, 1 = off (one step after another), else 4, 8, 16 or 32.
                                    Results are bit-identical either way.                              */
    int32_t host_threads;        /* shipsim_step_host: host threads that rebuild the observation rows (the caller included).
                                    0 = min(16, hardware threads); with several ranks on one box pass
                                    hardware threads / ranks so that the ranks do not oversubscribe the cores  */
} shipsim_config;

/* num_envs up to which steps_in_flight = 0 selects the time-parallel kernel (measured on B200, profiles/) */
#define SHIPSIM_WINDOW_AUTO_MAX_ENVS 32768

typedef struct shipsim_handle shipsim_t;

int shipsim_abi_version(void);
const char *shipsim_last_error(void);

/* Fill *cfg with the reference defaults (config.py:14-24, models.py:29,87,107, game.py:82,270,274-275). */
int shipsim_config_default(shipsim_config *cfg);

/* Replaces ShipEnv.__init__ / ShipGame.__init__ (ship_env.py:23-48, game.py:32-58) for a batch of envs. */
int shipsim_create(const shipsim_config *cfg, int device, shipsim_t **out);
int shipsim_destroy(shipsim_t *h);

/* Level data.  Replaces ShipGame.gen_level / PolyEnv / pm.Poly plane construction (game.py:60-71,
 * models.py:158-196) and the goal list of gen_goal_path (game.py:300-330): the host generates scenarios in
 * float64 (ship_sim_gym_b200/scenario.py) and hands over, per scenario, the two bank hulls (CCW, convex,
 * <= SHIPSIM_MAX_HULL vertices, host_hull_xy[s][bank][maxv][2], host_hull_n[s][bank]) and the 5 goal centres
 * (host_goals_xy[s][5][2]).  The vertices are rounded to fp32 and copied to the device, where the planes are derived
 * from them in double and packed as for a device-generated bank (the copy is owned by the handle).  Synchronous; call
 * once per curriculum change, not per step. */
int shipsim_load_scenarios(shipsim_t *h, const double *host_hull_xy, const int32_t *host_hull_n,
                           const double *host_goals_xy, int32_t n_scenarios, int32_t maxv);

/* The same level data generated ON THE DEVICE, replacing the host loop over ShipGame.reset() calls: per scenario
 * game_map.gen_river_poly (game_map.py:22-73; map_N segments per bank, bank width = width_frac * W / 2), pm.Poly's
 * convex hull (models.py:180) and ShipGame.gen_goal_path (game.py:300-330), in double precision, then the packing,
 * reach grid and spawn rows shipsim_load_scenarios derives.  Draws come from Philox4x32-10 keyed by (seed, scenario):
 * the distributions are the reference's, the individual maps are not (CPython's Mersenne Twister cannot be matched).
 * Work is enqueued on `stream`; the call waits for it (a 4-byte read-back sizes the SAT pass). */
int shipsim_generate_scenarios(shipsim_t *h, int32_t n_scenarios, uint64_t seed, int32_t map_N, float width_frac, void *stream);

/* Fresh maps in the reset path (ShipGame.reset builds a new level for every episode: game.py:271-272, game_map.py:22-73).
 * With enable != 0 the device-generated bank (shipsim_generate_scenarios; 4 * 2^k scenarios; auto_reset on) is treated as
 * four slices: resets of period p -- a period lasts at least max_steps env-steps, so an episode ends no later than the
 * period after the one it began in -- pick from slice p % 4, walking it with a per-env offset and odd stride (an env
 * does not meet a map twice), while the slice two periods ahead is regenerated with a new seed on a side stream.  No
 * map is played again once its slice has been retired.  enable == 0 returns to the fixed bank. */
int shipsim_fresh_maps(shipsim_t *h, int32_t enable);
/* info[8] = enabled, period, first scenario and size of the slice resets pick from, regeneration count of the 4 slices. */
int shipsim_fresh_info(const shipsim_t *h, int32_t *info);

/* Weighted scenario picks: resets (automatic and shipsim_reset without explicit scenarios) draw map i with probability
 * w[i] / sum(w) instead of uniformly, e.g. to hold maps out of training (weight 0) or to replay the maps a policy still
 * fails on.  dev_weights = uint32 w[n_scenarios] in DEVICE memory; the handle's table (prefix sums and a guide table, 8
 * bytes per scenario, allocated with the bank) is rebuilt from it by one kernel enqueued on `stream`: no allocation, no
 * synchronisation, so the call may sit between the replays of a captured CUDA graph, whose step launches then read the
 * new table.  The pick stays keyed by (seed, global env id, episode): equal weights give exactly the uniform picks, and
 * the draws do not depend on how the envs are sharded.  Where every weight is 0, or the weights sum to 2^32 or more,
 * the picks are uniform.  dev_weights == NULL returns to uniform picks.  A new bank (shipsim_load_scenarios,
 * shipsim_generate_scenarios) drops the weights.  Fresh maps (shipsim_fresh_maps) never replay a map, so the two exclude
 * each other: weights while fresh maps are on, and fresh maps while weights are on, fail with SHIPSIM_ERR_STATE. */
int shipsim_scenario_weights(shipsim_t *h, const uint32_t *dev_weights, void *stream);

/* Read the device-generated bank back (validation / inspection): host_hull_xy[n][2][SHIPSIM_MAX_HULL][2] (CCW, zero
 * padded), host_hull_n[n][2], host_goals[n][5][2]; hull vertices are the fp32-rounded ones the kernels use. */
int shipsim_read_scenarios(shipsim_t *h, double *host_hull_xy, int32_t *host_hull_n, double *host_goals);

/* Curriculum knob (ship_gym/curriculum.py:23-50 is meant to schedule scalars such as EnvConfig.MAX_STEPS, config.py:16):
 * change the episode length cap of a live handle.  Takes effect from the next shipsim_step; envs whose step count is
 * already at or beyond the new cap end on their next step, exactly as ShipEnv.is_done would (ship_env.py:131). */
int shipsim_set_max_steps(shipsim_t *h, int32_t max_steps);

/* Per-env state lives in ONE caller-owned device buffer of shipsim_state_bytes() bytes, laid out as
 * SHIPSIM_STATE_PLANES planes of float4[num_envs] (structure of arrays, 128 B per env):
 *   0: x, y, angle, vx          1: vy, w, episode_return, bits{rudder/5+2 | alive<<3 | step_count<<8}
 *   2: lidar[0..3]              3: lidar[4..7]            4: lidar[8], lidar[9], bits(scenario), bits(episode)
 *   5: goal0.xy, goal1.xy       6: goal2.xy, goal3.xy     7: goal4.xy, 0, 0
 * (readings past a fan of fewer than 10 beams are unused), then for lidar_beams > 10 ceil((lidar_beams - 10) / 4) more
 * planes: 8 + q holds lidar[10 + 4q .. 13 + 4q].
 * dev_stats: shipsim_stats_bytes() bytes of scratch for the episode statistics (zeroed by bind). */
size_t shipsim_state_bytes(const shipsim_t *h);
size_t shipsim_stats_bytes(const shipsim_t *h);
int shipsim_bind_state(shipsim_t *h, void *dev_state, void *dev_stats, void *stream);

/* Replaces ShipEnv.reset (ship_env.py:171-184) / ShipGame.reset (game.py:260-277).
 * dev_mask: uint8[num_envs], non-zero = reset that env (NULL = all).  dev_scenario: int32[num_envs] scenario
 * ids to use (NULL = Philox(seed, global env id, episode)).  first != 0 restarts the episode counter at 0.
 * dev_obs (optional): float[num_envs][(6 + lidar_beams) * history] receives the reset observation of the envs that were
 * reset: [-1 x (6 + lidar_beams) | x, y, 0, 0, gx, gy, -1 x lidar_beams] for history 2. */
int shipsim_reset(shipsim_t *h, const uint8_t *dev_mask, const int32_t *dev_scenario, int first, float *dev_obs,
                  void *stream);

/* Replaces ShipEnv.step (ship_env.py:136-156) for all envs, K consecutive steps in ONE launch.
 * dev_actions: [K][num_envs] of `action_dtype`, values in {0,1,2} (Discrete(3), ship_env.py:19; anything else
 * is treated like the decoder's no-op, game.py:152-153 -- range checking is the host layer's AssertionError).
 * Outputs, each [K][num_envs] leading: dev_obs float[..][(6 + lidar_beams) * history] (16-byte aligned for 10 beams, 4-byte
 * otherwise: the rows are dense), dev_reward float, dev_done uint8.  Any output pointer may be NULL to skip it. */
int shipsim_step(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs,
                 float *dev_reward, uint8_t *dev_done, void *stream);

/* shipsim_step for back-to-back rollouts: same arguments, same results, but a window-kernel launch may start while the
 * handle's previous launch still runs, each env waiting only for its own previous launch (a launch otherwise lasts as
 * long as its slowest warp).  It chains -- and counts in shipsim_chained_count -- when all of these hold:
 *   - the handle's previous call was a window-kernel launch on the same stream, and no ABI call of any handle enqueued
 *     work since (every other call that enqueues work, shipsim_step_host included, starts a new chain);
 *   - lidar_beams = 10, no episode log bound, fresh maps off;
 *   - the stream is not being captured into a graph.
 * Otherwise it is exactly shipsim_step.  Launch N + 1 still completes after launch N: whatever is enqueued later on the
 * stream sees both finished.  The caller promises that nothing enqueued on `stream` since the handle's previous step call
 * writes what this call reads (the actions), and that no kernel in between lets later launches start early (programmatic
 * dependent launch) while it reads what this call writes. */
int shipsim_step_chained(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs,
                         float *dev_reward, uint8_t *dev_done, void *stream);

/* Episode log.  With auto_reset a done env's observation is replaced by the reset observation; with a log bound, the
 * step kernels first append one record per finished episode: dev_meta[i][SHIPSIM_EPISODE_META] (SHIPSIM_EP_*) and
 * dev_rows[i][(6 + lidar_beams) * history] = exactly the row an auto_reset = 0 launch writes for that env at that step (terminal
 * observation; history = the config's 1 or 2).  Slots are reserved with an atomic add on *dev_count (int32, the records
 * appended so far); a record whose slot is >= capacity is not written, but the count keeps counting, so a caller sees
 * the loss.  The caller owns the three buffers (device memory; dev_rows and dev_meta may also be page-locked host
 * memory, written over PCIe without atomics -- dev_count must be device memory) and drains the log by reading it and
 * zeroing *dev_count on its stream.  SHIPSIM_EP_K includes the chunk offset on the chunked shipsim_step_host path;
 * SHIPSIM_EP_CALL counts shipsim_step / shipsim_step_host calls of the handle (a replayed CUDA graph repeats the
 * captured values).  Results with the log on are bit-identical to results with it off.  capacity == 0 unbinds.  Needs
 * auto_reset (SHIPSIM_ERR_STATE otherwise). */
int shipsim_episode_log_bind(shipsim_t *h, float *dev_rows, int32_t *dev_meta, int32_t capacity, int32_t *dev_count);

/* Same transition with HOST buffers: host_actions in, rows / rewards / done flags out, waited for (what a CPU-side caller
 * such as the reference's own training scripts sees).  Any output pointer may be NULL.  Buffers should be page-locked
 * (cudaHostAlloc / torch pin_memory); pageable ones work, more slowly.  How the bytes travel depends on the size of the
 * call: up to 64 KB of rows with page-locked buffers -- no copies, the kernel works on the caller's (mapped) memory; small
 * calls -- plain copies on `stream`; large ones with HISTORY_SIZE = 2 -- frames compacted on the device (~22 bytes per
 * env-step over PCIe) and expanded into the rows by `host_threads` host threads, optionally with a share of the envs as
 * complete rows by DMA (INTEGRATION.md); the compacted format is that of 10-beam frames, so other fans use the first two
 * regimes at every size.  host_obs[K][num_envs][(6 + lidar_beams) * history].  The results are identical bit for bit in
 * every case. */
int shipsim_step_host(shipsim_t *h, const int32_t *host_actions, int32_t K, float *host_obs, float *host_reward,
                      uint8_t *host_done, void *stream);

/* The host half of shipsim_step_host, exposed for callers that move frames themselves (and for the CPU tests): build
 * HISTORY_SIZE = 2 observation rows (ship_env.py:112-113) from 10-beam (16-float) frames.  host_frames holds the frame of the state before
 * the first step for every env (num_envs x 16 floats) followed by one 16-float frame per row, rows ordered [step][env];
 * host_obs[row] = [host_frames[row] | host_frames[row + num_envs]], except that where host_cut[row] != 0 (may be NULL)
 * the first half is 16 x -1: the observation ShipEnv.reset returns (ship_env.py:180-184).  Pure host code, no device. */
int shipsim_assemble_history(float *host_obs, const float *host_frames, const uint8_t *host_cut, int64_t n_rows, int64_t num_envs);

/* The host half of the compacted wire format shipsim_step_host uses for HISTORY_SIZE = 2 and 10-beam frames (exposed for callers that move
 * the data themselves, and for the CPU tests).  Per env-step a 16-byte record {bits(x), bits(y), bits(angle), word} with
 * word = (rudder / 5 + 2) | reward code << 3 (0 = step penalty, 1 = +1, 2 = -1) | done << 5 | change mask << 8, where bit j
 * of the mask says that slot 4 + j of the frame (gx, gy, lidar 0..9; ship_env.py:108-110) differs from the env's previous
 * frame; the changed values follow in host_var, those of the 32 envs of block b at step k starting at
 * host_off[k * ceil(num_envs / 32) + b], in env order then slot order.  host_cur[num_envs][16] holds the frame before
 * the first step on entry and the frame after the last on exit.  Outputs (any may be NULL): host_obs[n_steps][num_envs]
 * [16 * history], host_reward, host_done; with history = 2 and cut_on_done, a row whose done flag is set gets 16 x -1 as
 * its previous frame (ship_env.py:180-184).  Pure host code, no device. */
int shipsim_expand_delta(float *host_obs, float *host_reward, uint8_t *host_done, const uint32_t *host_rec, const uint32_t *host_off,
                         const float *host_var, float *host_cur, int32_t n_steps, int64_t num_envs, float step_penalty,
                         int32_t cut_on_done, int32_t history);

/* The policy half of an on-device rollout step (BASELINE configs[4]): stable-baselines' MlpPolicy as the reference trains it
 * (train/stable_baselines/ppo.py:88: separate tanh trunks obs -> 64 -> 64 for the policy and the value function, heads of 3
 * logits and 1 value) for num_envs observation rows of 32 floats, and the categorical sample by Gumbel-max.  fp32, one launch.
 * Layouts (device memory, row-major): dev_w1[32][128] = [policy | value] first layers side by side (any observation scale
 * folded in), dev_b1[128]; dev_w2[2][64][64] = the trunks' second layers (in x out), dev_b2[128]; dev_w3[128][4] = policy head in
 * rows 0..63 x columns 0..2, value head in rows 64..127 x column 3 (the other entries are not read), dev_b3[4];
 * dev_noise[num_envs][3] Gumbel(0, 1) draws.  Outputs: dev_out[num_envs][4] = 3 logits | value, dev_actions[num_envs] =
 * argmax(logits + noise) as int64 -- the dtype shipsim_step takes as SHIPSIM_ACTION_I64; the first maximum wins a tie.
 * Alignment: dev_obs, dev_w1, dev_b1, dev_w2, dev_b2, dev_w3 and dev_out 16 bytes, dev_actions 8 bytes (SHIPSIM_ERR_ARG
 * otherwise; dev_b3 and dev_noise need only float alignment).  Enqueued on `stream` on the current device. */
int shipsim_mlp_policy_forward(const float *dev_obs, int32_t num_envs, const float *dev_w1, const float *dev_b1, const float *dev_w2,
                               const float *dev_b2, const float *dev_w3, const float *dev_b3, const float *dev_noise, float *dev_out,
                               int64_t *dev_actions, void *stream);

/* Generalised advantage estimation over a finished rollout, as the PPO2 runner the reference trains with computes it
 * (train/stable_baselines/ppo.py:88,104): dev_rewards[T][N], dev_values[T + 1][N] (the last row = V of the observation after
 * the rollout), dev_dones[T][N] -> dev_adv[T][N], dev_returns[T][N] = adv + V.  One launch, enqueued on `stream`. */
int shipsim_gae(const float *dev_rewards, const float *dev_values, const uint8_t *dev_dones, int32_t n_steps, int32_t num_envs, float gamma,
                float lam, float *dev_adv, float *dev_returns, void *stream);

/* shipsim_gae over a rollout of the handle's envs (num_envs of them), plus the map every step played and Prioritized Level
 * Replay's value-loss scores per map.  The rollout is the handle's step calls call0, call0 + 1, ... (SHIPSIM_EP_CALL), each
 * of steps_per_call steps: the episode-log record of call c, step k is rollout step (c - call0) * steps_per_call + k.
 * Walking each env backwards from the last step, the steps after its last done belong to the scenario of the bound state
 * (the episode it plays now), and the steps up to and including a done at t to the scenario of the record of (t, env).
 * dev_adv / dev_returns are bit-identical to shipsim_gae's.  dev_step_scenario[T][num_envs] receives the scenario of every
 * step, -1 where the episode's record was lost (log capacity) -- those steps go to row n_scenarios of dev_scores.
 * dev_scores[n_scenarios + 1][SHIPSIM_SCORE_COLS] (doubles, ADDED into: zero it to start a table) sums per map the steps,
 * max(adv, 0) and |adv|; the sums are double atomics, so their last bits depend on the order the atomics land in.  The
 * record count is read on the device: no synchronisation, enqueued on `stream`, CUDA-graph capturable.  A replayed graph
 * repeats its captured call0, exactly as the records repeat their captured call numbers (SHIPSIM_EP_CALL), so the two stay
 * consistent.  Records of other calls are ignored.  Needs a bound state, a bank, auto_reset and an episode log
 * (SHIPSIM_ERR_STATE otherwise); the log must not be drained between the rollout's steps and this call. */
int shipsim_gae_scored(shipsim_t *h, const float *dev_rewards, const float *dev_values, const uint8_t *dev_dones, int32_t n_steps, float gamma,
                       float lam, int32_t call0, int32_t steps_per_call, float *dev_adv, float *dev_returns, int32_t *dev_step_scenario,
                       double *dev_scores, void *stream);

/* Reduce the per-CTA statistic slots into dev_out[SHIPSIM_STATS_LEN] doubles (device memory, e.g. the tensor
 * handed to ncclAllReduce); clear != 0 zeroes the slots afterwards.  Replaces the counters ShipEnv keeps on the
 * Python object (ship_env.py:150,152,177). */
int shipsim_stats_read(shipsim_t *h, double *dev_out, int clear, void *stream);

/* State injection / extraction for parity tests and checkpointing (SURVEY.md §5: the env has no save/restore in
 * the reference).  Host arrays, row-major: pose[n][6] = x y angle vx vy w; ints[n][5] = rudder, alive_mask,
 * step_count, scenario, episode; lidar[n][lidar_beams]; goals[n][5][2]; ep_return[n].  Synchronous. */
int shipsim_set_state(shipsim_t *h, const float *host_pose, const int32_t *host_ints, const float *host_lidar,
                      const float *host_goals, const float *host_ep_return);
int shipsim_get_state(shipsim_t *h, float *host_pose, int32_t *host_ints, float *host_lidar, float *host_goals,
                      float *host_ep_return);

/* Debug rendering of ONE env into dev_rgb[height][width][3] (uint8, device memory): replaces ShipGame.render +
 * get_screen (game.py:133-138,197-229), i.e. the `rgb_array` mode ShipEnv.metadata lists (ship_env.py:18).  Blue
 * background, banks, remaining goals, the hull, a circle per lidar ray where it ended (red = has hit, green = full
 * length) and the yellow position marker; screen y points down as in pygame.  Enqueued on `stream`. */
int shipsim_render(shipsim_t *h, int32_t env_index, int32_t width, int32_t height, uint8_t *dev_rgb, void *stream);

/* Introspection for benchmarks: launches issued so far, lanes per env and CTA size actually used. */
int shipsim_launch_count(const shipsim_t *h, int64_t *out);
int shipsim_launch_shape(const shipsim_t *h, int32_t *lanes_per_env, int32_t *threads_per_cta, int32_t *ctas);
/* bytes the last shipsim_step_host moved over PCIe (host->device actions; device->host frames / rows, rewards, dones) */
int shipsim_host_traffic(const shipsim_t *h, int64_t *h2d_bytes, int64_t *d2h_bytes);
/* host threads shipsim_step_host uses to rebuild observation rows (0 until its first call creates the pool) */
int shipsim_host_threads(const shipsim_t *h, int32_t *n_threads);
/* steps of one env the last launch speculated together (1 = the serial-in-time kernel ran) */
int shipsim_launch_window(const shipsim_t *h, int32_t *steps_in_flight);
/* shipsim_step_chained calls that chained onto the previous launch */
int shipsim_chained_count(const shipsim_t *h, int64_t *out);

#ifdef __cplusplus
}
#endif
#endif /* SHIPSIM_H */
