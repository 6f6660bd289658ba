/* level_oracle.c -- the CPU oracle (oracle/pgtg_oracle.c, included unmodified) with level sets. TEST INFRASTRUCTURE ONLY.
 *
 * A second opinion on the product's level sets (include/pgtg_b200.h, pgtg_levels): the pool is built with the oracle's own
 * generator (level j = the map generate_map builds for seed start_level + j at episode 1, the first after a seeded reset),
 * and every reset takes the episode's level and start square from the level block philox(counter = (0, 0, k,
 * PGTG_STREAM_LEVEL), seed) -- word 0 -> level (w0 * M) >> 32, or (env_id_base + i) mod M in env_index sampling; word 1 ->
 * the start square. Everything else -- the map build, the tick, traffic, observations, state -- is the oracle's code. */
#include "../../oracle/pgtg_oracle.c"

/* one level: the MapPlan generate_map returned for it */
typedef struct {
  unsigned char exits[PGTG_MAX_TILES], otype[PGTG_MAX_TILES], omask[PGTG_MAX_TILES];
  int sx, sy, sdir, gx, gy, gdir;
} lvl_level;

typedef struct {
  ora_batch base; /* first member: an lvl_batch* is an ora_batch* for the oracle's own functions */
  lvl_level* pool;
} lvl_batch;

static int level_of(const ora_batch* b, const ora_env* e, int64_t gid, uint32_t episode, uint32_t* start_word) {
  uint32_t blk[4] = {0u, 0u, episode, (uint32_t)PGTG_STREAM_LEVEL};
  philox4x32_10(blk, (uint32_t)e->seed, (uint32_t)(e->seed >> 32));
  if (start_word) *start_word = blk[1];
  int64_t M = b->cfg.num_levels;
  if (b->cfg.level_sampling) return (int)(((gid % M) + M) % M);
  return (int)(((uint64_t)blk[0] * (uint64_t)M) >> 32);
}

static void build_pool(lvl_batch* lb) {
  ora_batch* b = &lb->base;
  int M = b->cfg.num_levels;
  lb->pool = (lvl_level*)calloc((size_t)M, sizeof(lvl_level));
  ora_env* t = (ora_env*)calloc(1, sizeof(ora_env));
  for (int j = 0; j < M; j++) {
    memset(t, 0, sizeof *t);
    t->seed = (uint64_t)b->cfg.start_level + (uint64_t)j; t->episode = 1; t->blk_stream = -1; t->cblk_slot = -2;
    rctx r = {b, t};
    generate_map(&r, t);
    lvl_level* l = &lb->pool[j];
    memcpy(l->exits, t->exits, sizeof l->exits); memcpy(l->otype, t->otype, sizeof l->otype); memcpy(l->omask, t->omask, sizeof l->omask);
    l->sx = t->sx; l->sy = t->sy; l->sdir = t->sdir; l->gx = t->gx; l->gy = t->gy; l->gdir = t->gdir;
  }
  free(t);
}

static void load_level(ora_batch* b, ora_env* e, const lvl_level* l) {
  e->W = b->cfg.map_w; e->H = b->cfg.map_h;
  memcpy(e->exits, l->exits, sizeof e->exits); memcpy(e->otype, l->otype, sizeof e->otype); memcpy(e->omask, l->omask, sizeof e->omask);
  e->sx = l->sx; e->sy = l->sy; e->sdir = l->sdir; e->gx = l->gx; e->gy = l->gy; e->gdir = l->gdir;
}

/* env_reset of the oracle with map_path = this episode's level and the level block's start square */
static void lvl_env_reset(lvl_batch* lb, ora_env* e, int64_t gid) {
  ora_batch* b = &lb->base;
  rctx r = {b, e};
  e->episode++;
  e->elapsed = 0;
  memset(e->draw_k, 0, sizeof e->draw_k); e->blk_stream = -1; e->cblk_slot = -2;
  uint32_t start_word;
  load_level(b, e, &lb->pool[level_of(b, e, gid, e->episode, &start_word)]);
  build_episode_map(b, e);
  e->individual_subgoal_reward = b->cfg.sum_subgoals_reward / (double)e->num_subgoals;
  int si = (int)(((uint64_t)start_word * (uint64_t)e->n_starters) >> 32);
  if (e->n_starters > 0) { e->x = e->starters[si][0]; e->y = e->starters[si][1]; } else { e->x = e->y = 0; e->error |= 64; }
  e->vx = e->vy = 0;
  e->terminated = e->truncated = e->flat_tire = 0;
  e->n_cars = 0; e->next_car_id = 0; e->light_counter = 0;
  e->braking_applied = 0;
  e->outcome = 0;
  e->ep_return = 0;
  if (e->visited) {
    memset(e->visited, 0, (size_t)(e->width + 2) * (e->height + 2));
    e->visited[vis_index(e, e->x, e->y)] = 1;
  }
  if (b->cfg.traffic_density > 0) create_initial_traffic(&r);
}

/* reset_job / step_job of the oracle with lvl_env_reset */
static void* lvl_reset_job(void* p) {
  job* j = (job*)p; ora_batch* b = j->b;
  size_t os = (size_t)b->C * b->P * b->P;
  for (int i = j->lo; i < j->hi; i++) {
    if (j->mask && !j->mask[i]) continue;
    ora_env* e = &b->envs[i];
    if (j->seeds) { e->seed = (uint64_t)j->seeds[i]; e->episode = 0; }
    lvl_env_reset((lvl_batch*)b, e, b->cfg.env_id_base + i);
    if (j->obs_map) get_observation(b, e, j->obs_map + os * i, j->obs_pos + 2 * i, j->obs_vel + 2 * i, j->obs_nsd + i);
  }
  return NULL;
}

static void* lvl_step_job(void* p) {
  job* j = (job*)p; ora_batch* b = j->b;
  size_t os = (size_t)b->C * b->P * b->P;
  for (int i = j->lo; i < j->hi; i++) {
    ora_env* e = &b->envs[i];
    double cost = 0;
    double rew = env_step(b, e, j->actions[i], &cost);
    e->ep_return += rew;
    int trunc = b->cfg.max_episode_steps > 0 && e->elapsed >= b->cfg.max_episode_steps;
    j->reward[i] = rew; j->cost[i] = cost;
    j->terminated[i] = (uint8_t)e->terminated; j->truncated[i] = (uint8_t)trunc;
    j->step_state[4 * i] = e->x; j->step_state[4 * i + 1] = e->y; j->step_state[4 * i + 2] = e->vx; j->step_state[4 * i + 3] = e->vy;
    j->step_flags[i] = (uint8_t)((e->flat_tire ? 1 : 0) | (e->braking_applied ? 2 : 0));
    if (e->terminated || trunc) {
      if (j->f_map) get_observation(b, e, j->f_map + os * i, j->f_pos + 2 * i, j->f_vel + 2 * i, j->f_nsd + i);
      j->stats[0] += 1; j->stats[1] += e->ep_return; j->stats[2] += e->elapsed;
      if (e->terminated) { if (e->outcome == 2) j->stats[3] += 1; else j->stats[4] += 1; }
      else j->stats[5] += 1;
      lvl_env_reset((lvl_batch*)b, e, b->cfg.env_id_base + i);
    }
    get_observation(b, e, j->obs_map + os * i, j->obs_pos + 2 * i, j->obs_vel + 2 * i, j->obs_nsd + i);
  }
  return NULL;
}

ora_batch* lvl_create(const pgtg_config* cfg) {
  if (cfg->num_levels < 1 || cfg->rng_mode != PGTG_RNG_PHILOX || cfg->fixed_map) return NULL;
  lvl_batch* lb = (lvl_batch*)calloc(1, sizeof *lb);
  ora_batch* b = &lb->base;
  b->cfg = *cfg;
  b->N = cfg->num_envs; b->C = cfg->num_channels; b->P = cfg->sliding ? 2 * cfg->window_k + 1 : 9;
  b->threads = 1;
  build_pool(lb);
  return b;
}

int lvl_reset(ora_batch* b, const int64_t* seeds, const uint8_t* mask, int8_t* obs_map, int32_t* obs_pos, int32_t* obs_vel, int32_t* obs_nsd) {
  if (ensure_envs(b)) return -1;
  job j; memset(&j, 0, sizeof j);
  j.b = b; j.seeds = seeds; j.mask = mask; j.obs_map = obs_map; j.obs_pos = obs_pos; j.obs_vel = obs_vel; j.obs_nsd = obs_nsd;
  run_jobs(b, &j, lvl_reset_job);
  return 0;
}

int lvl_step(ora_batch* b, const int32_t* actions, int8_t* obs_map, int32_t* obs_pos, int32_t* obs_vel, int32_t* obs_nsd, double* reward,
             double* cost, uint8_t* terminated, uint8_t* truncated, int32_t* step_state, uint8_t* step_flags, int8_t* f_map, int32_t* f_pos,
             int32_t* f_vel, int32_t* f_nsd) {
  if (!b->envs) return -1;
  job j; memset(&j, 0, sizeof j);
  j.b = b; j.actions = actions; j.obs_map = obs_map; j.obs_pos = obs_pos; j.obs_vel = obs_vel; j.obs_nsd = obs_nsd;
  j.reward = reward; j.cost = cost; j.terminated = terminated; j.truncated = truncated;
  j.step_state = step_state; j.step_flags = step_flags; j.f_map = f_map; j.f_pos = f_pos; j.f_vel = f_vel; j.f_nsd = f_nsd;
  run_jobs(b, &j, lvl_step_job);
  return 0;
}

/* level of every env's current (previous = 0) or previous episode */
int lvl_levels(ora_batch* b, int32_t* out, int previous) {
  if (!b->envs) return -1;
  for (int i = 0; i < b->N; i++) out[i] = level_of(b, &b->envs[i], b->cfg.env_id_base + i, b->envs[i].episode - (uint32_t)(previous != 0), NULL);
  return 0;
}

/* the pool in the layout of pgtg_dlpack's "level_tiles" (uint16 [M, T], with the subgoal directions build_episode_map
 * derives) and "level_plan" (uint32 [M], plan word of pgtg_device.cuh, start-square bits clear) */
int lvl_pool(ora_batch* b, uint16_t* tiles, uint32_t* plan) {
  lvl_batch* lb = (lvl_batch*)b;
  int T = b->cfg.map_w * b->cfg.map_h;
  ora_env* t = (ora_env*)calloc(1, sizeof *t);
  if (!t || !env_alloc(b, t)) return -2;
  for (int j = 0; j < b->cfg.num_levels; j++) {
    const lvl_level* l = &lb->pool[j];
    load_level(b, t, l);
    build_episode_map(b, t);
    for (int k = 0; k < T; k++) {
      int sg = t->tile_dir[k] >= 0 ? t->tile_dir[k] + 1 : 0;
      tiles[(size_t)j * T + k] = (uint16_t)(l->exits[k] | l->otype[k] << 4 | l->omask[k] << 7 | sg << 11);
    }
    plan[j] = (uint32_t)l->sx | (uint32_t)l->sy << 4 | (uint32_t)l->sdir << 8 | (uint32_t)l->gx << 10 | (uint32_t)l->gy << 14 |
              (uint32_t)l->gdir << 18 | (uint32_t)t->num_subgoals << 20;
  }
  free(t->grid); free(t->sq_type); free(t->starters); free(t->spawnable); free(t->spawners); free(t->cars); free(t->visited); free(t);
  return 0;
}

void lvl_destroy(ora_batch* b) {
  if (!b) return;
  free(((lvl_batch*)b)->pool);
  ora_destroy(b);  /* frees the envs and the batch allocation itself (the lvl_batch: base is its first member) */
}
