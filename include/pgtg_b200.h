/* pgtg_b200 -- C ABI of the B200-native batched PGTG simulator.
 *
 * The reference (Inuri04/pgtg) has no FFI: its hot path sits behind the Gymnasium Env API of
 * `PGTGEnv` (pgtg/environment.py:297). This header is that API, batched, as plain C:
 *
 *   reference call                                   replaced by
 *   ------------------------------------------------ ---------------------------------------
 *   PGTGEnv.__init__(**kwargs)  environment.py:302   pgtg_create(const pgtg_config*, ...)
 *   json_file_to_map_plan       parser.py:227        pgtg_load_fixed_map
 *   PGTGEnv.reset(seed=...)     environment.py:581   pgtg_reset
 *   PGTGEnv.step(action)        environment.py:1092  pgtg_step (device actions) /
 *                                                    pgtg_step_host (host buffers, e2e)
 *   PGTGEnv.get_observation     environment.py:1344  written by pgtg_step/pgtg_reset into the
 *                                                    buffers returned by pgtg_get_buffers
 *   PGTGEnv.get_info            environment.py:1538  step_* buffers + pgtg_get_state
 *   PGTGEnv.set_to_state        environment.py:1301  pgtg_set_state
 *   np_random draws             environment.py:593   pgtg_load_draws (conformance) / Philox
 *
 * All functions return 0 on success or a negative pgtg_status; pgtg_last_error() gives the
 * thread-local message. No exceptions and no torch types cross this boundary. All device work
 * is enqueued on the caller-supplied CUDA stream (a cudaStream_t passed as void*); only the
 * *_host / get_state / stats calls synchronise. One handle per GPU; calls on one handle must be
 * serialised by the caller (the reference is single-threaded too).
 */
#ifndef PGTG_B200_H
#define PGTG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGTG_ABI_VERSION 2
#define PGTG_MAX_CHANNELS 16
#define PGTG_MAX_RULES 8
#define PGTG_NUM_PROFILES 5
#define PGTG_NUM_ROUTE_IDS 20
#define PGTG_MAX_TILES 256 /* map_w * map_h */

typedef enum pgtg_status {
  PGTG_OK = 0,
  PGTG_ERR_INVALID = -1, /* bad argument / config (ValueError on the Python side) */
  PGTG_ERR_CUDA = -2,    /* CUDA runtime failure (RuntimeError) */
  PGTG_ERR_STATE = -3,   /* call order / mode misuse (RuntimeError) */
  PGTG_ERR_DRAWS = -4    /* conformance tape exhausted or tag mismatch */
} pgtg_status;

/* Observation plane kinds (environment.py:1387-1445). The host maps feature names to kinds. */
typedef enum pgtg_channel {
  PGTG_CH_ZERO = 0,        /* a literal feature name no square ever carries */
  PGTG_CH_WALLS = 1,       /* "walls" (:1389) / literal "wall"; off-map = wall when sliding */
  PGTG_CH_GOALS = 2,       /* "goals" = subgoal | final goal (:1392) */
  PGTG_CH_TRAFFIC = 3,     /* "traffic": car positions (:1397) */
  PGTG_CH_ICE = 4,
  PGTG_CH_BROKEN = 5,
  PGTG_CH_SAND = 6,
  PGTG_CH_LIGHT_GREEN = 7, /* only via the literal "traffic_light" entry (:1411-1439) */
  PGTG_CH_LIGHT_YELLOW = 8,
  PGTG_CH_LIGHT_RED = 9,
  PGTG_CH_SUBGOAL = 10,    /* literal names matched by the generic loop (:1441-1445) */
  PGTG_CH_FINAL_GOAL = 11,
  PGTG_CH_START = 12,
  PGTG_CH_USED_SUBGOAL = 13,
  PGTG_CH_CAR_SPAWNER = 14
} pgtg_channel;

/* Random-number source. */
typedef enum pgtg_rng_mode {
  PGTG_RNG_PHILOX = 0, /* counter-based Philox4x32-10 per env (production) */
  PGTG_RNG_TAPE = 1,   /* conformance: consume draws recorded from the reference's np_random */
  PGTG_RNG_NUMPY = 2   /* numpy-exact: SeedSequence + PCG64 + Generator.random/integers/choice restated, so
                          that seeds alone reproduce the reference (env i = SeedSequence(seed_i)) */
} pgtg_rng_mode;

/* Draw tags on a conformance tape: stream * 8 + kind. */
enum { PGTG_STREAM_MAP = 0, PGTG_STREAM_CAR = 1, PGTG_STREAM_ICE = 2, PGTG_STREAM_BROKEN = 3, PGTG_STREAM_SAND = 4 };
/* Philox counter word 3 of the level draw (level sets, pgtg_levels); never a tape tag */
enum { PGTG_STREAM_LEVEL = 5 };
enum { PGTG_DRAW_DOUBLE = 0, PGTG_DRAW_INDEX = 1 };

/* Agent heading ids used by traffic rules (environment.py:185-206). */
enum { PGTG_AGENT_S2N = 0, PGTG_AGENT_W2E = 1, PGTG_AGENT_N2S = 2, PGTG_AGENT_E2W = 3, PGTG_AGENT_STATIONARY = 4, PGTG_AGENT_NEAR_GOAL = 5 };

/* One TrafficRule (environment.py:130-159), flattened. */
typedef struct pgtg_rule {
  int32_t tile_type;    /* exits N | E<<1 | S<<2 | W<<3 of rule.tile_type, -1 = never matches */
  int32_t min_traffic;
  int32_t min_matching_traffic;
  int32_t reserved;
  double vel_lo, vel_hi; /* velocity_range, compared with sqrt(vx^2+vy^2) */
  /* weight[a][r] = number of maneuvers with agent==a whose traffic list contains route r */
  uint8_t weight[6][PGTG_NUM_ROUTE_IDS];
} pgtg_rule;

/* PGTGEnv.__init__ keyword arguments (environment.py:302-359), frozen into a POD. Quantities the
 * reference computes with Python semantics (banker's round(), cumsum/normalise, float products)
 * are computed on the host and passed as numbers so that device code never re-derives them. */
typedef struct pgtg_config {
  int32_t abi_version;
  int32_t num_envs;
  int64_t env_id_base; /* global id of local env 0 (multi-GPU shards keep global streams) */
  uint64_t seed;       /* Philox base seed; env i uses seed + env_id_base + i */
  int32_t rng_mode;    /* pgtg_rng_mode */
  int32_t fixed_map;   /* 1: map comes from pgtg_load_fixed_map (map_path), 0: procedural */

  /* procedural map (map_generator.py:43-472) */
  int32_t map_w, map_h;        /* random_map_width / height, tiles */
  int32_t edges_to_keep;       /* round(len(removable_edges) * pct), directed count (:242) */
  int32_t border_connections;  /* round(len(possible) * pct) (:362-364) */
  int32_t start_mode, goal_mode; /* 0: (x,y,dir) given, 1: (x,y) given, 2: "random" */
  int32_t start_x, start_y, start_dir, goal_x, goal_y, goal_dir; /* normalised (no -1), dir N0 E1 S2 W3 */
  int32_t min_start_goal_distance; /* -1 = None */
  int32_t num_levels;  /* level set: 0 = every episode gets a fresh map; M in 1..2^24 = episodes draw one of M pre-built
                          maps (pgtg_levels). Philox mode, procedural maps only */
  double obstacle_probability;
  double obstacle_cdf[4]; /* cumsum(p)/cumsum(p)[-1] for ice, broken road, sand, traffic_light */

  /* observation (environment.py:417-441, 1344-1506) */
  int32_t num_channels;
  int32_t channel_kind[PGTG_MAX_CHANNELS];
  int32_t sliding;   /* use_sliding_observation_window */
  int32_t window_k;  /* sliding_observation_window_size (also used by the rule engine, :1061) */
  int32_t use_next_subgoal_direction;

  /* rewards (environment.py:340-345) */
  double sum_subgoals_reward, final_goal_bonus, crash_penalty, traffic_light_violation_penalty;
  double standing_still_penalty, already_visited_position_penalty;
  /* obstacle trigger probabilities (:346-348) */
  double ice_probability, street_damage_probability, sand_probability;
  /* traffic (:349-357) */
  double traffic_density;
  int32_t light_green, light_yellow, light_red; /* traffic_light_phases_duration */
  int32_t ignore_traffic_collisions;
  double profile_cdf[PGTG_NUM_PROFILES]; /* conservative, normal, aggressive, elderly, reckless */
  /* DRIVER_BEHAVIORS (environment.py:64-109), with the derived thresholds as host doubles */
  double drv_yellow_stop[PGTG_NUM_PROFILES];
  double drv_red_violation[PGTG_NUM_PROFILES];
  double drv_patience_threshold[PGTG_NUM_PROFILES]; /* patience_level * 10   (:954) */
  double drv_push_probability[PGTG_NUM_PROFILES];   /* 1.0 - patience_level  (:956) */
  double drv_speed_multiplier[PGTG_NUM_PROFILES];
  double drv_reaction_delay[PGTG_NUM_PROFILES];
  int32_t drv_min_following[PGTG_NUM_PROFILES];
  int32_t separate_reward_cost;

  int32_t num_rules;
  int32_t level_sampling; /* with num_levels: 0 = uniform draw per episode, 1 = env (env_id_base + i) keeps level (env_id_base + i) mod M */
  pgtg_rule rules[PGTG_MAX_RULES];

  /* vector-env additions (the reference gets these from wrappers: train.py:39) */
  int32_t max_episode_steps;  /* TimeLimit; 0 = none */
  int32_t write_final_obs;    /* 1: also write the terminal observation of done envs */
  int32_t max_cars;           /* capacity per env; 0 = derive from 32*W*H*density */
  int32_t start_level;        /* with num_levels: level j is the first map of key start_level + j (0 .. 2^31 - 1) */
} pgtg_config;

/* One tile of a fixed map plan (MapPlan.tiles[y][x], map_generator.py:10-17). */
typedef struct pgtg_tile {
  uint8_t exits;         /* N | E<<1 | S<<2 | W<<3 */
  uint8_t obstacle_type; /* 0 none, 1 ice, 2 broken road, 3 sand, 4 traffic_light */
  uint8_t obstacle_mask; /* mask id 0..13 (see pgtg_tables.h) */
  uint8_t reserved;
} pgtg_tile;

/* Device buffers owned by the handle; valid until pgtg_destroy. Shapes in elements. */
typedef struct pgtg_buffers {
  int32_t num_envs, num_channels, window; /* window = P (9 or 2k+1) */
  int32_t max_cars;
  int8_t* obs_map;         /* [N, C, P, P], cell index [x][y] (environment.py:1529-1534) */
  int32_t* obs_position;   /* [N, 2] */
  int32_t* obs_velocity;   /* [N, 2] */
  int32_t* obs_next_subgoal_direction; /* [N] (-1 when disabled) */
  double* reward;          /* [N] */
  double* cost;            /* [N] safety cost when separate_reward_cost, else 0 */
  uint8_t* terminated;     /* [N] */
  uint8_t* truncated;      /* [N] */
  /* outcome of the tick itself (terminal values for envs that were auto-reset) */
  int32_t* step_state;     /* [N, 4] x, y, vx, vy */
  uint8_t* step_flags;     /* [N] bit0 flat_tire, bit1 braking_applied */
  /* terminal observation of auto-reset envs (only when write_final_obs) */
  int8_t* final_obs_map;           /* [N, C, P, P] or NULL */
  int32_t* final_obs_position;     /* [N, 2] or NULL */
  int32_t* final_obs_velocity;     /* [N, 2] or NULL */
  int32_t* final_obs_next_subgoal_direction; /* [N] or NULL */
  /* episode statistics accumulated on device: episodes, sum_return, sum_length, goals,
   * crashes, truncations, sum of discounted returns, negative discounted returns (the last two with
   * pgtg_set_evaluation; doubles so one NCCL all-reduce(sum) covers them) */
  double* stats;           /* [8] */
} pgtg_buffers;

/* Host-side snapshot of every env's state (parity dumps, set_to_state). Arrays are caller-owned,
 * sized [N] / [N, max_cars] / [N, map_w*map_h]; any pointer may be NULL to skip that field. */
typedef struct pgtg_state {
  int32_t* agent;      /* [N, 4] x, y, vx, vy */
  uint8_t* flat_tire;  /* [N] */
  int32_t* light_counter; /* [N] */
  int32_t* elapsed;    /* [N] ticks since reset */
  int32_t* num_cars;   /* [N] */
  int32_t* cars;       /* [N, max_cars, 7] id, x, y, route, profile, patience, delay */
  uint16_t* tiles;     /* [N, T] exits | type<<4 | mask<<7 | sgdir<<11 (0 none, 1+dir) */
  int32_t* plan;       /* [N, 8] sx, sy, sdir, gx, gy, gdir, num_subgoals, reserved */
  uint8_t* used;       /* [N, T] subgoal of tile consumed */
  int64_t* draw_cursor; /* [N] tape cursor (conformance) */
  int32_t* error;      /* [N] sticky per-env error flags (tape mismatch etc.) */
} pgtg_state;

typedef struct pgtg_env pgtg_env;

const char* pgtg_last_error(void);
int pgtg_abi_version(void);

int pgtg_create(const pgtg_config* cfg, int device, pgtg_env** out);
int pgtg_destroy(pgtg_env* env);

/* tiles[y * w + x]; start/goal as (x, y, dir). Requires cfg.fixed_map. */
int pgtg_load_fixed_map(pgtg_env* env, const pgtg_tile* tiles, int w, int h,
                        int sx, int sy, int sdir, int gx, int gy, int gdir);

/* (2R+1)^2 host-generated direction LUT: low 3 bits = compass octant of atan2(dy,dx)
 * (environment.py:1069-1088), bits 3-5 = remapped index of atan2(-dy,dx) (:1486-1502);
 * entry index (dy + R) * (2R+1) + (dx + R). Generated with the host's libm so the device never
 * evaluates atan2. */
int pgtg_load_direction_lut(pgtg_env* env, const uint8_t* lut, int radius);

/* Conformance tape (host arrays): values[offsets[i] .. offsets[i+1]) are env i's draws in program
 * order, tags[j] = stream*8 + kind. Index draws are stored as integral doubles. */
int pgtg_load_draws(pgtg_env* env, const double* values, const uint8_t* tags,
                    const int64_t* offsets);

/* Reset envs (mask == NULL: all; else host uint8[N]). seeds (host int64[N]) may be NULL to keep
 * each env's current stream (a later reset() without seed, environment.py:593-599). */
int pgtg_reset(pgtg_env* env, const int64_t* seeds, const uint8_t* mask, void* stream);

/* One tick for every env, with same-step auto-reset. actions: device int32[N] (or int64 when
 * action_bytes == 8). No host synchronisation. */
int pgtg_step(pgtg_env* env, const void* actions_dev, int action_bytes, void* stream);

/* The same tick through host buffers (copies inside): actions int32[N] in; any out pointer may
 * be NULL. This is the call a non-CUDA host (the reference-facing plugin) makes. */
int pgtg_step_host(pgtg_env* env, const int32_t* actions, int8_t* obs_map, int32_t* obs_position,
                   int32_t* obs_velocity, double* reward, uint8_t* terminated, uint8_t* truncated,
                   void* stream);

/* The same with the observation planes as BITS (env i at bit i * C*P*P of obs_packed, pgtg_packed_obs_bytes bytes in
 * all: 92 B per env instead of 729 at the defaults) and the copies double-buffered on a copy stream: the tick of the next
 * call does not wait for this call's device-to-host copies. wait != 0 returns when the host buffers are complete;
 * wait == 0 leaves them in flight until pgtg_host_sync. pgtg_unpack_obs turns the bits back into int8 cells on the host. */
int64_t pgtg_packed_obs_bytes(pgtg_env* env);
int pgtg_step_host_packed(pgtg_env* env, const int32_t* actions, uint32_t* obs_packed, int32_t* obs_position, int32_t* obs_velocity,
                          double* reward, uint8_t* terminated, uint8_t* truncated, int wait, void* stream);
int pgtg_host_sync(pgtg_env* env);
int pgtg_unpack_obs(const uint32_t* obs_packed, int8_t* obs_map, int64_t n_cells, int threads);

/* Observation format (call before the first pgtg_reset; PGTG_ERR_STATE after it, PGTG_ERR_INVALID for an unknown format).
 * PGTG_OBS_INT8, the default: every tick writes obs_map (and final_obs_map) as int8 cells. PGTG_OBS_BITS: every tick
 * stores the planes only as bits, to the device buffer "obs_packed" (uint32 [ceil(N * C*P*P / 32)], env i at bit i * C*P*P,
 * the layout of pgtg_step_host_packed) and, with write_final_obs, terminal observations to "final_obs_packed" (same layout;
 * rows of envs that did not finish are not meaningful). obs_map and final_obs_map stay allocated but are written only by
 * pgtg_expand_obs. Scalars, pgtg_step_host, pgtg_step_host_packed, pgtg_flatten, pgtg_observe, checkpoints (which then
 * carry the bits: a blob of one format does not load into a handle of the other) and level sets work as in int8. */
#define PGTG_OBS_INT8 0
#define PGTG_OBS_BITS 1
int pgtg_set_obs_format(pgtg_env* env, int format);
/* Bits format: expand obs_packed (final != 0: final_obs_packed) into obs_map (final_obs_map) on `stream`, no synchronisation. */
int pgtg_expand_obs(pgtg_env* env, int final, void* stream);
/* Rows of stored bits -> int8 cells or the flattened float32 observation, on `stream`, no synchronisation (either format of
 * the handle). bits_dev: `slots` step slots back to back, pgtg_packed_obs_bytes each (a [slots, words] tensor of obs_packed
 * copies); row r = s * N + i is env i of slot s. index_dev: device int64 [count] rows, or NULL for rows 0 .. count - 1.
 * PGTG_UNPACK_INT8: out_dev int8 [count, C, P, P] (32-byte aligned), cells as in obs_map. PGTG_UNPACK_FLAT: out_dev float32
 * [count, D] in the order of pgtg_flatten (plane_order: host int32 [C], as there), position_dev / velocity_dev int32
 * [slots, N, 2] and nsd_dev int32 [slots, N] (when next_subgoal_direction is on) gathered with the same rows. A row
 * outside [0, slots * N) gives an all-zero output row and sets error flag 256 (pgtg_error_summary). */
#define PGTG_UNPACK_INT8 0
#define PGTG_UNPACK_FLAT 1
int pgtg_unpack_bits(pgtg_env* env, const uint32_t* bits_dev, int64_t slots, const int64_t* index_dev, int64_t count, int format,
                     void* out_dev, const int32_t* plane_order, const int32_t* position_dev, const int32_t* velocity_dev,
                     const int32_t* nsd_dev, void* stream);

/* Recompute the observation buffers from the current state without ticking (the second half of
 * set_to_state, environment.py:1342). */
int pgtg_observe(pgtg_env* env, void* stream);

/* add_traffic_rule / remove_traffic_rule (environment.py:569-575): replace the rule table. */
int pgtg_update_rules(pgtg_env* env, const pgtg_rule* rules, int num_rules);

int pgtg_get_buffers(pgtg_env* env, pgtg_buffers* out);
/* DLPack export of one buffer of pgtg_buffers by field name ("obs_map", "reward", ...): *out
 * receives a DLManagedTensor* (DLPack v0 ABI) that the caller wraps in a PyCapsule named
 * "dltensor" (or hands to any DLPack consumer). The memory stays owned by the handle; the
 * deleter only frees the descriptor. */
int pgtg_dlpack(pgtg_env* env, const char* name, void** out_managed_tensor);
int pgtg_get_state(pgtg_env* env, pgtg_state* out);
/* The computed parts of PGTGEnv.get_info (environment.py:1538-1578), host arrays, any pointer may be NULL:
 * agent_direction int32[N] = index into {south_to_north, west_to_east, north_to_south, east_to_west, stationary,
 * near_goal} (get_agent_direction_string, :185-206); current_tile_type int32[N] = exits N | E<<1 | S<<2 | W<<3 of the
 * agent's tile (:1541-1549); profile_counts int32[N, 5] = cars per driver profile (get_driver_profile_stats,
 * :1017-1035). Synchronises. */
int pgtg_get_info(pgtg_env* env, int32_t* agent_direction, int32_t* current_tile_type, int32_t* profile_counts);
/* set_to_state (environment.py:1301-1342): agent, flat_tire and cars only (quirk A.3-10). */
int pgtg_set_state(pgtg_env* env, const pgtg_state* in);
/* Full-state checkpoint / clone (PGTGEnv.light_step deep-copies the env, environment.py:1283-1299; the reference's
 * set_to_state restores only a part, quirk A.3-10): everything a tick reads or writes -- SoA state, both ring slots and the
 * map-request queues, car lists, RNG state / tape cursors, light counters, patience and delays, consumed subgoals, episode
 * statistics and the output buffers. save/load go through a host blob of pgtg_state_bytes bytes; copy is device to device
 * between two handles of the same configuration on the same device. All three synchronise. */
int64_t pgtg_state_bytes(pgtg_env* env);
int pgtg_save_state(pgtg_env* env, void* out, int64_t out_bytes);
int pgtg_load_state(pgtg_env* env, const void* in, int64_t in_bytes);
int pgtg_copy_state(pgtg_env* dst, pgtg_env* src);
/* Evaluator statistics (ModularEvaluator.evaluate, evaluator.py:292-339): gamma > 0 switches on the per-env discounted
 * return (total += reward * pow(gamma, t), the powers evaluated on the host), zeroes the running discounted returns and
 * sets the episode cap to max_steps; stats[6] = sum of the discounted returns of the finished episodes, stats[7] = how
 * many of them were negative (terminated = stats[3] + stats[4], over max_steps = stats[5]). gamma <= 0 switches it off
 * and restores the configured cap (max_episode_steps of the configuration, or the one pgtg_copy_state took from its
 * source). Evaluation does not change the state layout: blobs and copies stay compatible with handles that never
 * evaluated, and they do not carry the discounted returns of episodes in flight (loading or copying zeroes them).
 * Synchronises. */
int pgtg_set_evaluation(pgtg_env* env, double gamma, int max_steps);
/* Episode statistics are accumulated per CTA on the device. pgtg_reduce_stats sums them into the
 * 8-double `stats` buffer on `stream` without synchronising (so the host can NCCL-all-reduce that
 * device buffer); pgtg_reset_stats clears them. */
int pgtg_reduce_stats(pgtg_env* env, void* stream);
int pgtg_reset_stats(pgtg_env* env, void* stream);
/* Reduces, then copies the 8 statistics doubles to the host (synchronises). */
int pgtg_stats(pgtg_env* env, double* out8, int reset_after);
/* Flattened float32 observation [N, D] in gymnasium 0.28.1 FlattenObservation order over the reference's
 * Dict space (train.py:39-40): sorted map planes, next_subgoal_direction one-hot (if enabled), position
 * one-hots, velocity. plane_order[i] = channel index of the i-th plane in sorted-key order. The buffer is
 * allocated on first use, owned by the handle and also exported as DLPack "obs_flat". */
int pgtg_flatten(pgtg_env* env, const int32_t* plane_order, void* stream, float** out_dev, int* out_dim);

/* Level sets (num_levels > 0). Level j (0 <= j < M) is the map -- tiles, obstacles, start, goal, subgoal path -- that a
 * handle without levels gives an env of key start_level + j at its first episode after a seeded reset; the pool is built
 * once by pgtg_create and exported through pgtg_dlpack as "level_tiles" (uint16 [M, T], descriptor layout of
 * pgtg_state.tiles) and "level_plan" (uint32 [M], packed start / goal / subgoal count, start-square bits clear). Episode k
 * of env i draws its level and start square from one block philox(counter = (0, 0, k, PGTG_STREAM_LEVEL), key_i):
 * word 0 -> level (w0 * M) >> 32 (uniform; env_index sampling uses (env_id_base + i) mod M instead), word 1 -> start
 * square (w1 * 3) >> 32 when the start line is labelled "start" (else error flag 64). pgtg_levels writes every env's level
 * as device int32[N] on `stream` without synchronising: of the current episode (previous = 0) or of the one before it
 * (previous = 1: for an env that auto-reset in the last step, the episode that just ended). */
int pgtg_levels(pgtg_env* env, int32_t* out_dev, int previous, void* stream);

/* Per-kernel device timing: while enabled (max_steps > 0), pgtg_step brackets each of its kernels
 * with CUDA events on the launching stream; pgtg_timing synchronises and returns the summed
 * durations in ms of the tick kernel and of the map-generation kernel over the recorded ticks. */
int pgtg_enable_timing(pgtg_env* env, int max_steps);
/* Map generation normally overlaps the next tick (side stream, small persistent grid). on = 0 runs the two
 * kernels back to back on the caller's stream instead, e.g. to time each kernel alone. Synchronises. */
int pgtg_set_overlap(pgtg_env* env, int on);
int pgtg_timing(pgtg_env* env, double* tick_ms, double* mapgen_ms, int* steps);
/* OR of every env's sticky error flags (bit 7 = 128: an action outside 0..8 was replaced by the no-op 4, where the
 * reference raises KeyError; the other bits are listed in pgtg_api_impl.hpp) and of the handle's (bit 8 = 256: a
 * pgtg_unpack_bits index out of range). Synchronises. */
int pgtg_error_summary(pgtg_env* env, uint32_t* out_flags);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t pgtg_launch_count(pgtg_env* env);
/* Which kernel instantiations a step of this handle launches, as text ("tick=traffic(G=32,NT=256) ..."). */
int pgtg_kernel_info(pgtg_env* env, char* out, int out_bytes);

#ifdef __cplusplus
}
#endif
#endif /* PGTG_B200_H */
