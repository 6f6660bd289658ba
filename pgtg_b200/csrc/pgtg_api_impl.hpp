// pgtg_api_impl.hpp -- implementation of the C ABI (include/pgtg_b200.h) over a small memory /
// launch backend. Included exactly once by
//   pgtg_b200/csrc/pgtg_kernels.cu   backend = CUDA runtime on sm_100a (the product), and
//   tests/emu/pgtg_emu.cpp           backend = host memory + loops (CPU test-suite only).
// The including file defines, before the #include:
//   void* bk_alloc(size_t);  void bk_free(void*);  int bk_set_device(int);
//   int bk_h2d(void* dst, const void* src, size_t n, void* stream);   (async on stream)
//   int bk_d2h(void* dst, const void* src, size_t n, void* stream);   (async on stream)
//   int bk_memset(void* dst, int v, size_t n);  int bk_memset_async(void*, int, size_t, void* stream);  int bk_sync(void* stream);
//   int bk_launch(pgtg_env*, int mode, const uint8_t* mask_dev, const int64_t* seeds_dev,
//                 const void* actions_dev, int action_bytes, void* stream);
//   const char* bk_error();  int bk_dl_device_type();
//   int bk_conn_table_max_bits();  int bk_build_conn_table(pgtg_env*, uint32_t* table_dev);
//   int bk_build_path_table(pgtg_env*, uint64_t* table_dev);
//   bool bk_inline_mapgen();   whether the backend has the tick instantiation that generates maps itself (PGTG_INLINE_MAPGEN)
//   int bk_side_create(void** stream, void** ev_tick, void** ev_map0, void** ev_map1, int* sm_count);
//   void bk_side_destroy(void*, void*, void*, void*);  int bk_stream_wait(void* stream, void* ev);
//   void* bk_event_create();  void bk_event_destroy(void*);  int bk_event_record(void* ev, void* stream);
//   double bk_event_elapsed(void* a, void* b);
//   int bk_stats_reduce(pgtg_env*, void* stream);  int bk_stats_reset(pgtg_env*, void* stream);
//   int bk_d2d(void* dst, const void* src, size_t n, void* stream);  void* bk_stream_create();  void bk_stream_destroy(void*);
//   int bk_info(pgtg_env*, int32_t* out_dev);  int bk_error_or(pgtg_env*, uint32_t* out_dev);   (*out_dev = OR of p.error[0..N))   (info_env for every env)
//   void bk_traffic_geometry(const DevCfg&, int* G, int* NT);   (G = 0: the traffic tick cannot run this configuration)
#pragma once
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "pgtg_phases.cuh"

using namespace pgtg;

#include "pgtg_env.hpp"

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }

extern "C" const char* pgtg_last_error(void) { return g_err.c_str(); }
extern "C" int pgtg_abi_version(void) { return PGTG_ABI_VERSION; }

template <typename T>
static T* dev_alloc(pgtg_env* e, size_t count, bool zero = true) {
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  void* ptr = bk_alloc(bytes);
  if (!ptr) return nullptr;
  e->allocs.push_back(ptr);
  if (zero) bk_memset(ptr, 0, bytes);
  return (T*)ptr;
}

// removable_edges order = graph-theory Graph.edges() after the add_edge calls of
// generate_map_graph (map_generator.py:218-227): nodes in first-mention order, each node's
// successors in insertion order. Node = tile index y * W + x.
static void build_edge_tables(int W, int H, std::vector<uint16_t>& tab, std::vector<uint16_t>& rev) {
  int T = W * H;
  std::vector<int> order;
  std::vector<char> known(T, 0);
  std::vector<std::vector<int>> nbr(T);
  auto add = [&](int a, int b) {
    if (!known[a]) { known[a] = 1; order.push_back(a); }
    if (!known[b]) { known[b] = 1; order.push_back(b); }
    nbr[a].push_back(b);
    nbr[b].push_back(a);  // bidirectional=True: reverse edge right after the forward one
  };
  for (int x = 0; x < W; x++)
    for (int y = 0; y < H; y++) {
      if (x < W - 1) add(y * W + x, y * W + x + 1);
      if (y < H - 1) add(y * W + x, (y + 1) * W + x);
    }
  tab.clear();
  for (int a : order) for (int b : nbr[a]) tab.push_back((uint16_t)(a | b << 8));
  rev.assign(tab.size(), 0);
  for (size_t i = 0; i < tab.size(); i++)
    for (size_t j = 0; j < tab.size(); j++)
      if ((tab[j] & 255) == (tab[i] >> 8) && (tab[j] >> 8) == (tab[i] & 255)) rev[i] = (uint16_t)j;
}

// possible_connections_to_borders (map_generator.py:350-360): rows (tile_y, tile_x, dir), with the
// DEFAULT start and goal slots removed whatever the actual start/goal are
static void build_border_slots(int W, int H, std::vector<uint16_t>& slots) {
  struct Row { int y, x, d; };
  std::vector<Row> rows;
  for (int x = 0; x < W; x++) rows.push_back({0, x, 0});
  for (int y = 0; y < H; y++) rows.push_back({y, W - 1, 1});
  for (int x = 0; x < W; x++) rows.push_back({H - 1, x, 2});
  for (int y = 0; y < H; y++) rows.push_back({y, 0, 3});
  auto remove_first = [&](int y, int x, int d) {
    for (size_t i = 0; i < rows.size(); i++)
      if (rows[i].y == y && rows[i].x == x && rows[i].d == d) { rows.erase(rows.begin() + i); return; }
  };
  remove_first(H - 1, 0, 3);
  remove_first(0, W - 1, 1);
  slots.clear();
  for (auto& r : rows) slots.push_back((uint16_t)((r.y * W + r.x) | r.d << 8));
}

// direction table evaluated with the host libm (the CPython `math` module calls the same atan2);
// see pgtg_load_direction_lut in the header
static void build_direction_lut(int R, std::vector<uint8_t>& lut) {
  int n = 2 * R + 1;
  lut.assign((size_t)n * n, 0);
  const double PI_8 = M_PI / 8;
  static const int remap[8] = {2, 1, 0, 7, 6, 5, 4, 3};
  for (int dy = -R; dy <= R; dy++)
    for (int dx = -R; dx <= R; dx++) {
      double a = atan2((double)dy, (double)dx);
      int o;
      if (-PI_8 <= a && a < PI_8) o = 2;
      else if (PI_8 <= a && a < 3 * PI_8) o = 3;
      else if (3 * PI_8 <= a && a < 5 * PI_8) o = 4;
      else if (5 * PI_8 <= a && a < 7 * PI_8) o = 5;
      else if (a >= 7 * PI_8 || a < -7 * PI_8) o = 6;
      else if (-7 * PI_8 <= a && a < -5 * PI_8) o = 7;
      else if (-5 * PI_8 <= a && a < -3 * PI_8) o = 0;
      else o = 1;
      double a2 = atan2((double)(-dy), (double)dx);
      int idx = (int)fmod((a2 + M_PI) / (M_PI / 4), 8.0);
      lut[(size_t)(dy + R) * n + (dx + R)] = (uint8_t)(o | remap[idx & 7] << 3);
    }
}

// CTA size of the tick kernel: the largest of 128 / 64 / 32 envs whose shared memory fits 200 KB (a wide sliding window
// with many planes, or a large map, outgrows it at 128), or PGTG_BLOCK when that fits. Both backends run the
// CTA decomposition this picks, so the emulation covers the device's smaller CTAs too.
static int pick_block(const DevCfg& c, int* block, size_t* smem) {
  const char* forced = getenv("PGTG_BLOCK");  // experiment knob: CTA size of the tick kernel (32 / 64 / 128)
  int fb = forced ? atoi(forced) : 0;
  if (fb == 32 || fb == 64 || fb == 128) {
    size_t s = block_shared_bytes(c, fb);
    if (s <= 200 * 1024) { *block = fb; *smem = s; return 0; }
  }
  for (int B : {128, 64, 32}) {
    size_t s = block_shared_bytes(c, B);
    if (s <= 200 * 1024) { *block = B; *smem = s; return 0; }
  }
  return -1;
}

// The plain configuration the LEAN tick instantiation promises (pgtg_logic.cuh, env_step): decided at
// pgtg_create and again whenever something it depends on changes (pgtg_update_rules, pgtg_set_state).
static int lean_predicate(const pgtg_config& c, const DevCfg& d) {
  const bool plain = d.pregen && !(c.traffic_density > 0) && !d.rules_without_traffic && d.kind_channel[PGTG_CH_CAR_SPAWNER] < 0 && !d.vis_words &&
                     !c.separate_reward_cost && (c.sliding || d.obs_fast);
  if (!plain) return 0;
  return (c.sliding || d.use_nsd) ? 2 : 1;  // 2: the lean SLIDE instantiation (terminal observations: the FINAL ones)
}

// The LUT block the kernels stage into shared memory: the generated tables plus everything derived from them.
static const LutInit h_lut_init = {PGTG_TAB_WALL, PGTG_TAB_EXIT_LINE, PGTG_TAB_MASK, PGTG_TAB_LANE_ANY, PGTG_TAB_NATIVE_SPAWNER, PGTG_TAB_ENTRY_SQ};
static const uint64_t h_lane_desc[16][81] = PGTG_TAB_LANE_DESC;
static void derive_lut(Lut& L) {
  memset(&L, 0, sizeof L);
  memcpy(L.wall, h_lut_init.wall, sizeof L.wall); memcpy(L.exit_line, h_lut_init.exit_line, sizeof L.exit_line);
  memcpy(L.mask, h_lut_init.mask, sizeof L.mask); memcpy(L.lane_any, h_lut_init.lane_any, sizeof L.lane_any);
  memcpy(L.native_spawner, h_lut_init.native_spawner, sizeof L.native_spawner); memcpy(L.entry_sq, h_lut_init.entry_sq, sizeof L.entry_sq);
  // local columns that can hold a car_spawner: native spawners and tile-entry squares
  for (int e = 0; e < 16; e++) { int ns = L.native_spawner[e]; if (ns != 255) L.spawner_cols |= 1u << (ns / TILE); }
  for (int d = 0; d < 4; d++) L.spawner_cols |= 1u << (L.entry_sq[d] / TILE);
  for (int w = 0; w < 3; w++) L.exit_any[w] = L.exit_line[0][w] | L.exit_line[1][w] | L.exit_line[2][w] | L.exit_line[3][w];
  for (int d = 0; d < 4; d++) {
    int n = 0;
    for (int sq = 0; sq < 81; sq++) if (((L.exit_line[d][sq >> 5] >> (sq & 31)) & 1u) && n < 4) { L.line_xy[d][n] = (uint8_t)((sq / TILE) | (sq % TILE) << 4); L.line_sq[d][n++] = (uint8_t)sq; }
  }
  for (int e = 0; e < 16; e++) {
    L.lane_count[e] = (uint8_t)(__builtin_popcount(L.lane_any[e][0]) + __builtin_popcount(L.lane_any[e][1]) + __builtin_popcount(L.lane_any[e][2]));
    // border spawners: the tile-entry square carries 'car_lane all <inward>' (parser.py:120-148); slots 1..4 = north, east,
    // south, west border of the map <-> all down (2), all left (3), all up (1), all right (4) on entry_sq[1], [2], [0], [3]
    static const int sq_of[4] = {1, 2, 0, 3}, all_of[4] = {2, 3, 1, 4};
    for (int k = 0; k < 4; k++) if ((int)(h_lane_desc[e][L.entry_sq[sq_of[k]]] & 7) == all_of[k]) L.entry_ok[e] |= (uint8_t)(1u << k);
  }
}

static int fill_devcfg(const pgtg_config& c, DevCfg& d, std::string& why) {
  memset(&d, 0, sizeof d);
  if (c.abi_version != PGTG_ABI_VERSION) { why = "pgtg_config.abi_version mismatch"; return -1; }
  if (c.num_envs < 1) { why = "num_envs must be >= 1"; return -1; }
  if (c.map_w < 1 || c.map_h < 1 || c.map_w > 16 || c.map_h > 16) { why = "map width/height must be in 1..16 tiles"; return -1; }
  if (c.num_channels < 0 || c.num_channels > PGTG_MAX_CHANNELS) { why = "too many observation planes"; return -1; }
  if (c.sliding && (c.window_k < 0 || c.window_k > 15)) { why = "sliding_observation_window_size must be in 0..15"; return -1; }
  if (c.num_rules < 0 || c.num_rules > PGTG_MAX_RULES) { why = "too many traffic rules"; return -1; }
  if (c.light_green + c.light_yellow + c.light_red <= 0 || c.light_green + c.light_yellow + c.light_red > 0x3FFF) { why = "traffic light durations out of range"; return -1; }
  if (c.rng_mode != PGTG_RNG_PHILOX && c.rng_mode != PGTG_RNG_TAPE && c.rng_mode != PGTG_RNG_NUMPY) { why = "unknown rng_mode"; return -1; }
  if (c.max_cars > 0xFFFF) { why = "max_cars too large"; return -1; }
  d.N = c.num_envs; d.W = c.map_w; d.H = c.map_h; d.T = c.map_w * c.map_h; d.WS = c.map_w * TILE; d.HS = c.map_h * TILE;
  d.C = c.num_channels; d.P = c.sliding ? 2 * c.window_k + 1 : TILE; d.sliding = c.sliding; d.window_k = c.window_k;
  d.use_nsd = c.use_next_subgoal_direction;
  for (int i = 0; i < PGTG_MAX_CHANNELS; i++) d.channel_kind[i] = c.channel_kind[i];
  for (int k = 0; k < 16; k++) d.kind_channel[k] = -1;
  d.obs_fast = 1;
  for (int i = 0; i < c.num_channels; i++) {
    int k = c.channel_kind[i];
    if (k <= 0 || k >= 16) continue;  // PGTG_CH_ZERO planes stay zero
    if (d.kind_channel[k] >= 0) d.obs_fast = 0;  // listed twice: generic channel loop
    d.kind_channel[k] = i;
  }
  d.fixed_map = c.fixed_map; d.edges_to_keep = c.edges_to_keep; d.border_connections = c.border_connections;
  d.start_mode = c.start_mode; d.goal_mode = c.goal_mode;
  d.start_x = c.start_x; d.start_y = c.start_y; d.start_dir = c.start_dir;
  d.goal_x = c.goal_x; d.goal_y = c.goal_y; d.goal_dir = c.goal_dir; d.min_sg_dist = c.min_start_goal_distance;
  d.obstacle_probability = c.obstacle_probability;
  for (int i = 0; i < 4; i++) d.obstacle_cdf[i] = c.obstacle_cdf[i];
  d.sum_subgoals_reward = c.sum_subgoals_reward; d.final_goal_bonus = c.final_goal_bonus; d.crash_penalty = c.crash_penalty;
  d.light_penalty = c.traffic_light_violation_penalty; d.standing_penalty = c.standing_still_penalty;
  d.visited_penalty = c.already_visited_position_penalty;
  d.ice_p = c.ice_probability; d.broken_p = c.street_damage_probability; d.sand_p = c.sand_probability;
  d.traffic_density = c.traffic_density;
  d.light_green = c.light_green; d.light_yellow = c.light_yellow; d.light_total = c.light_green + c.light_yellow + c.light_red;
  d.ignore_traffic_collisions = c.ignore_traffic_collisions;
  for (int i = 0; i < 5; i++) {
    d.profile_cdf[i] = c.profile_cdf[i]; d.drv_yellow_stop[i] = c.drv_yellow_stop[i]; d.drv_red_violation[i] = c.drv_red_violation[i];
    d.drv_patience_threshold[i] = c.drv_patience_threshold[i]; d.drv_push_probability[i] = c.drv_push_probability[i];
    d.drv_speed_multiplier[i] = c.drv_speed_multiplier[i]; d.drv_reaction_delay[i] = c.drv_reaction_delay[i];
    d.drv_min_following[i] = c.drv_min_following[i];
  }
  d.separate_reward_cost = c.separate_reward_cost; d.num_rules = c.num_rules; d.max_episode_steps = c.max_episode_steps;
  d.write_final_obs = c.write_final_obs;
  for (int i = 0; i < c.num_rules; i++) if (c.rules[i].min_traffic <= 0 && c.rules[i].min_matching_traffic <= 0) d.rules_without_traffic = 1;
  d.max_cars = c.max_cars > 0 ? c.max_cars : 1;
  d.lut_radius = (d.WS > d.HS ? d.WS : d.HS) + 2;
  int words = (d.T + 1) / 2;
  if ((words & 1) == 0) words++;  // odd word stride: conflict-free shared-memory rows
  d.tile_stride = words * 2;
  for (int t = 0; t < d.T; t++) {
    if (t % d.W < d.W - 1) d.full_e[t >> 5] |= 1u << (t & 31);
    if (t + d.W < d.T) d.full_s[t >> 5] |= 1u << (t & 31);
  }
  if (c.already_visited_position_penalty != 0) { d.vis_w = d.HS + 2; d.vis_words = ((d.WS + 2) * (d.HS + 2) + 31) / 32; }
  d.obs_bits = d.C * d.P * d.P;
  if (c.traffic_density > 0) { d.occ_words = (d.WS * d.HS + 15) / 16;  /* 2-bit counters */ d.spawner_cap = 2 * (d.W + d.H) + d.T; }
  d.pregen = (c.rng_mode != PGTG_RNG_TAPE && !c.fixed_map) ? 1 : 0;
  d.lean = lean_predicate(c, d);
  d.env_id_base = c.env_id_base; d.seed = c.seed;
  if (!c.fixed_map) {
    d.n_edge_tab = 2 * (d.W * (d.H - 1) + d.H * (d.W - 1));
    d.n_border_slots = 2 * d.W + 2 * d.H - 2;
    // connectivity table: fixed start/goal, single-register boards, <= 24 undirected grid edges
    // (2^24 bits = 2 MB); the emulation build caps it lower to keep CPU tests fast
    int n_he = d.H * (d.W - 1), n_ve = d.W * (d.H - 1);
    if (c.start_mode == 0 && c.goal_mode == 0 && d.T <= 32 && n_he + n_ve >= 1 && n_he + n_ve <= bk_conn_table_max_bits() &&
        !(c.start_x == c.goal_x && c.start_y == c.goal_y)) {
      d.conn_bits = n_he + n_ve; d.conn_ne = n_he;
      d.path_tab = d.T <= 16 ? 1 : 0;  // 8 bytes per edge set: 128 MB for the 4x4 grid
    }
    int n_slots = 2 * d.W + 2 * d.H - 2;
    if (c.border_connections < 0 || c.border_connections > n_slots) { why = "random_map_percentage_of_connections must be in [0, 1]"; return -1; }
    if (c.edges_to_keep < 0) { why = "random_map_percentage_of_connections must be in [0, 1]"; return -1; }
  }
  return 0;
}

extern "C" int pgtg_create(const pgtg_config* cfg, int device, pgtg_env** out) {
  if (!cfg || !out) return fail(PGTG_ERR_INVALID, "null argument");
  *out = nullptr;
  DevCfg dc;
  std::string why;
  if (fill_devcfg(*cfg, dc, why)) return fail(PGTG_ERR_INVALID, why);
  if (bk_set_device(device)) return fail(PGTG_ERR_CUDA, std::string("cannot select device: ") + bk_error());
  pgtg_env* e = new pgtg_env();
  e->cfg = *cfg; e->dc = dc; e->device = device; e->launches = 0;
  e->have_fixed = e->have_tape = e->did_reset = false;
  e->cars_injected = false;
  e->timing = false; e->tev_used = 0;
  e->side_stream = e->ev_tick = e->ev_map[0] = e->ev_map[1] = nullptr;
  e->launch_index = 0; e->mapgen_grid = 0; e->inline_mapgen = false;
  e->flat = nullptr; e->flat_dim = 0;
  e->info_dev = nullptr;
  e->packed_dev = nullptr; e->stage_dev[0] = e->stage_dev[1] = nullptr; e->stage_bytes = 0; e->copy_stream = nullptr;
  e->ev_stage[0] = e->ev_stage[1] = e->ev_copied[0] = e->ev_copied[1] = nullptr; e->host_steps = 0;
  memset(&e->dp, 0, sizeof e->dp);
  if (pick_block(e->dc, &e->block, &e->smem)) { delete e; return fail(PGTG_ERR_INVALID, "observation window too large for shared memory"); }
  e->nblk = (dc.N + e->block - 1) / e->block;
  e->stats_rows = nullptr;
  e->traffic_G = e->traffic_NT = 0;
  // The traffic tick runs every Philox configuration with cars. (Car-free configurations outside the lean tick's promise --
  // sliding window, next_subgoal_direction -- stay on the general tick: measured 1.05e9 vs 5.1e8 env-steps/s at 1 M envs, the
  // traffic tick's phase structure costs more per env than it saves; PGTG_TRAFFIC_KERNEL_CARFREE=1 forces it for tests.)
  const bool wants_traffic_tick = cfg->traffic_density > 0 || ((cfg->sliding || cfg->use_next_subgoal_direction) && !cfg->fixed_map && getenv("PGTG_TRAFFIC_KERNEL_CARFREE"));
  if (cfg->rng_mode == PGTG_RNG_PHILOX && wants_traffic_tick && !getenv("PGTG_NO_TRAFFIC_KERNEL")) bk_traffic_geometry(e->dc, &e->traffic_G, &e->traffic_NT);
  e->stats_nrows = e->nblk;
  if (e->traffic_G > 0 && (dc.N + e->traffic_G - 1) / e->traffic_G > e->stats_nrows) e->stats_nrows = (dc.N + e->traffic_G - 1) / e->traffic_G;
  DevPtrs& p = e->dp;
  size_t N = (size_t)dc.N;
  bool ok = true;
#define A(field, type, count) ok = ok && ((p.field = dev_alloc<type>(e, (count))) != nullptr) && (e->state_allocs.push_back({p.field, sizeof(type) * (size_t)(count)}), true)
  A(agent, short4, N); A(misc, uint32_t, N); A(elapsed, uint32_t, N); A(episode, uint32_t, N); A(next_car_id, uint32_t, N);
  A(plan, uint32_t, N); A(tiles, uint16_t, N * dc.T + 8);
  if (dc.pregen) { A(next_tiles, uint16_t, 2 * N * dc.T + 8); A(next_plan, uint32_t, 2 * N); A(regen_list, uint2, 4 * N); A(regen_count, uint32_t, 4); } A(cars, uint64_t, 2 * (size_t)dc.max_cars * N);
  if (dc.vis_words) A(visited, uint32_t, (size_t)dc.vis_words * N);
  if (dc.occ_words) { A(occ, uint32_t, (size_t)dc.occ_words * N); A(spawners, uint16_t, (size_t)dc.spawner_cap * N); A(spawner_count, uint16_t, N); }
  A(key, uint64_t, N); A(error, uint32_t, N); A(ep_return, double, N);
  if (cfg->rng_mode == PGTG_RNG_TAPE) { A(cursor, int64_t, N); A(tape_end, int64_t, N); }
  if (cfg->rng_mode == PGTG_RNG_NUMPY) { A(pcg, PcgState, 4 * N); p.pcg_stride = N; }
  A(obs_map, int8_t, N * dc.obs_bits + 16); A(obs_position, int32_t, 2 * N); A(obs_velocity, int32_t, 2 * N); A(obs_nsd, int32_t, N);
  A(reward, double, N); A(cost, double, N); A(terminated, uint8_t, N); A(truncated, uint8_t, N);
  A(step_state, int32_t, 4 * N); A(step_flags, uint8_t, N);
  if (dc.write_final_obs) {
    A(f_obs_map, int8_t, N * dc.obs_bits + 16); A(f_obs_position, int32_t, 2 * N); A(f_obs_velocity, int32_t, 2 * N); A(f_obs_nsd, int32_t, N);
  }
  A(stats, double, 8);
  ok = ok && ((e->stats_rows = dev_alloc<double>(e, 8 * (size_t)e->stats_nrows)) != nullptr) && (e->state_allocs.push_back({e->stats_rows, 64 * (size_t)e->stats_nrows}), true);
  ok = ok && ((e->mask_dev = dev_alloc<uint8_t>(e, N)) != nullptr);
  ok = ok && ((e->seeds_dev = dev_alloc<int64_t>(e, N)) != nullptr);
  ok = ok && ((e->actions_dev = dev_alloc<int32_t>(e, N)) != nullptr);
#undef A
  if (!ok) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error()); }
  // next_subgoal_direction is -1 when the feature is off (environment.py:1358)
  {
    std::vector<int32_t> neg(N, -1);
    bk_h2d(p.obs_nsd, neg.data(), N * 4, nullptr);
    if (p.f_obs_nsd) bk_h2d(p.f_obs_nsd, neg.data(), N * 4, nullptr);
    std::vector<uint64_t> keys(N);
    for (size_t i = 0; i < N; i++) keys[i] = cfg->seed + (uint64_t)cfg->env_id_base + i;
    bk_h2d(p.key, keys.data(), N * 8, nullptr);
    bk_sync(nullptr);
  }
  // tables
  if (!cfg->fixed_map) {
    build_edge_tables(dc.W, dc.H, e->edge_tab, e->edge_rev);
    build_border_slots(dc.W, dc.H, e->border_slots);
    if (e->dc.n_edge_tab != (int)e->edge_tab.size() || e->dc.n_border_slots != (int)e->border_slots.size()) {
      pgtg_destroy(e);
      return fail(PGTG_ERR_INVALID, "internal: map table sizes");
    }
    for (size_t i = 0; i < e->edge_tab.size(); i++) {
      // bit of this (undirected) edge in the connectivity-table index: horizontal edges compressed row by
      // row (W - 1 per row), then the vertical edges by tile index
      int a = e->edge_tab[i] & 255, b = e->edge_tab[i] >> 8, lo = a < b ? a : b;
      bool horiz = (a > b ? a - b : b - a) == 1 && dc.W != 1;
      int pos = horiz ? (lo / dc.W) * (dc.W - 1) + lo % dc.W : dc.H * (dc.W - 1) + lo;
      e->edge_rev[i] = (uint16_t)(e->edge_rev[i] | (pos & 63) << 10);
    }
    uint16_t* t1 = dev_alloc<uint16_t>(e, e->edge_tab.size() + 1);
    uint16_t* t2 = dev_alloc<uint16_t>(e, e->edge_rev.size() + 1);
    uint16_t* t3 = dev_alloc<uint16_t>(e, e->border_slots.size() + 1);
    if (!t1 || !t2 || !t3) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, "device allocation failed"); }
    bk_h2d(t1, e->edge_tab.data(), e->edge_tab.size() * 2, nullptr);
    bk_h2d(t2, e->edge_rev.data(), e->edge_rev.size() * 2, nullptr);
    bk_h2d(t3, e->border_slots.data(), e->border_slots.size() * 2, nullptr);
    p.edge_tab = t1; p.edge_rev = t2; p.border_slots = t3;
  }
  {
    Lut L;
    derive_lut(L);
    Lut* ld = dev_alloc<Lut>(e, 1);
    if (!ld) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, "device allocation failed"); }
    bk_h2d(ld, &L, sizeof L, nullptr);
    bk_sync(nullptr);  // (L is a stack object)
    p.lut = ld;
    // the lane probe of a car inside a tile (environment.py:891-932) as a table: which of the four neighbour squares
    // that lie in the SAME tile continue the car's route in that direction (tile-crossing moves are looked up live)
    std::vector<uint8_t> sl((size_t)16 * 81 * PGTG_NUM_ROUTE_IDS, 0);
    static const int DX[4] = {0, 0, -1, 1}, DY[4] = {-1, 1, 0, 0};
    for (int ex = 0; ex < 16; ex++)
      for (int sq = 0; sq < 81; sq++)
        for (int dd = 0; dd < 4; dd++) {
          int nx = sq / TILE + DX[dd], ny = sq % TILE + DY[dd];
          if (nx < 0 || ny < 0 || nx >= TILE || ny >= TILE) continue;
          uint64_t l = h_lane_desc[ex][nx * TILE + ny];
          for (int r = 0; r < PGTG_NUM_ROUTE_IDS; r++) {
            uint8_t& v = sl[((size_t)ex * 81 + sq) * PGTG_NUM_ROUTE_IDS + r];
            if ((int)(l & 7) == dd + 1) v |= (uint8_t)(16u << dd);
            for (int i = 0; i < (int)((l >> 3) & 7); i++)
              if ((int)((l >> (6 + 7 * i)) & 31) == r && (int)((l >> (11 + 7 * i)) & 3) == dd) v |= (uint8_t)(1u << dd);
          }
        }
    // ... and the same question asked of a square of ANOTHER tile (the move crosses a tile border)
    std::vector<uint8_t> tl((size_t)16 * 81 * PGTG_NUM_ROUTE_IDS, 0);
    for (int ex = 0; ex < 16; ex++)
      for (int sq = 0; sq < 81; sq++) {
        uint64_t l = h_lane_desc[ex][sq];
        for (int r = 0; r < PGTG_NUM_ROUTE_IDS; r++) {
          uint8_t& v = tl[((size_t)ex * 81 + sq) * PGTG_NUM_ROUTE_IDS + r];
          if ((l & 7) != 0) v |= (uint8_t)(16u << ((l & 7) - 1));
          for (int i = 0; i < (int)((l >> 3) & 7); i++)
            if ((int)((l >> (6 + 7 * i)) & 31) == r) v |= (uint8_t)(1u << ((l >> (11 + 7 * i)) & 3));
        }
      }
    uint8_t* sd = dev_alloc<uint8_t>(e, sl.size());
    uint8_t* tdv = dev_alloc<uint8_t>(e, tl.size());
    if (!sd || !tdv) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, "device allocation failed"); }
    bk_h2d(sd, sl.data(), sl.size(), nullptr);
    bk_h2d(tdv, tl.data(), tl.size(), nullptr);
    bk_sync(nullptr);
    p.step_lut = sd; p.target_lut = tdv;
  }
  {
    std::vector<uint8_t> lut;
    build_direction_lut(dc.lut_radius, lut);
    uint8_t* d = dev_alloc<uint8_t>(e, lut.size());
    pgtg_rule* r = dev_alloc<pgtg_rule>(e, PGTG_MAX_RULES);
    if (!d || !r) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, "device allocation failed"); }
    bk_h2d(d, lut.data(), lut.size(), nullptr);
    bk_h2d(r, cfg->rules, sizeof(pgtg_rule) * PGTG_MAX_RULES, nullptr);
    p.dirlut = d; p.rules = r;
  }
  if (e->dc.pregen) {
    int sms = 0;
    if (bk_side_create(&e->side_stream, &e->ev_tick, &e->ev_map[0], &e->ev_map[1], &sms)) {
      pgtg_destroy(e);
      return fail(PGTG_ERR_CUDA, std::string("cannot create the map-generation stream: ") + bk_error());
    }
    const char* env_ctas = getenv("PGTG_MAPGEN_CTAS_PER_SM");
    int per_sm = env_ctas ? atoi(env_ctas) : 0;  // 0 = full grid (best with the connectivity table, see DESIGN.md 7)
    e->mapgen_grid = per_sm > 0 ? sms * per_sm : 0;
    e->mapgen_grid_overlap = e->mapgen_grid; e->overlap = !getenv("PGTG_NO_OVERLAP");
    e->inline_mapgen = bk_inline_mapgen() && getenv("PGTG_INLINE_MAPGEN") != nullptr && cfg->rng_mode == PGTG_RNG_PHILOX && !getenv("PGTG_NO_LEAN");  // (and map_in_registers: below)
  }
  if (e->dc.conn_bits) {
    size_t words = ((size_t)1 << e->dc.conn_bits) / 32 + 1;
    uint32_t* t = dev_alloc<uint32_t>(e, words, false);
    if (!t || bk_build_conn_table(e, t)) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, std::string("connectivity table: ") + bk_error()); }
    p.conn_table = t;
    // the grid faces next to every edge (remove_edges_tabled: an edge whose face is otherwise intact cannot disconnect anything)
    const int W = e->dc.W, H = e->dc.H, n_he = H * (W - 1);
    std::vector<uint2> ft((size_t)e->dc.conn_bits);
    for (auto& m : ft) m.x = m.y = 0x80000000u;
    auto add = [&](int edge, uint32_t others) { uint2& m = ft[(size_t)edge]; if (m.x == 0x80000000u) m.x = others; else m.y = others; };
    for (int r = 0; r + 1 < H; r++)
      for (int x = 0; x + 1 < W; x++) {
        const int f[4] = {r * (W - 1) + x, (r + 1) * (W - 1) + x, n_he + r * W + x, n_he + r * W + x + 1};  // top, bottom, left, right
        uint32_t all = 0;
        for (int k = 0; k < 4; k++) all |= 1u << f[k];
        for (int k = 0; k < 4; k++) add(f[k], all & ~(1u << f[k]));
      }
    uint2* fd = dev_alloc<uint2>(e, ft.size());
    if (!fd) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, "device allocation failed"); }
    bk_h2d(fd, ft.data(), ft.size() * sizeof(uint2), nullptr);
    p.face_tab = fd;
  }
  if (e->dc.path_tab) {
    uint64_t* t = dev_alloc<uint64_t>(e, (size_t)1 << e->dc.conn_bits, false);
    if (!t || bk_build_path_table(e, t)) { pgtg_destroy(e); return fail(PGTG_ERR_CUDA, std::string("path table: ") + bk_error()); }
    p.path_table = t;
  }
  if (!pgtg::map_in_registers(e->dc)) e->inline_mapgen = false;  // (needs both tables, decided just above)
  bk_sync(nullptr);
  *out = e;
  return PGTG_OK;
}

extern "C" int pgtg_destroy(pgtg_env* e) {
  if (!e) return PGTG_OK;
  bk_set_device(e->device);
  bk_side_destroy(e->side_stream, e->ev_tick, e->ev_map[0], e->ev_map[1]);
  bk_sync(nullptr);
  for (void* ev : e->tev) bk_event_destroy(ev);
  for (int i = 0; i < 2; i++) { if (e->ev_stage[i]) bk_event_destroy(e->ev_stage[i]); if (e->ev_copied[i]) bk_event_destroy(e->ev_copied[i]); }
  if (e->copy_stream) bk_stream_destroy(e->copy_stream);
  for (void* a : e->allocs) bk_free(a);
  delete e;
  return PGTG_OK;
}

extern "C" int pgtg_load_fixed_map(pgtg_env* e, const pgtg_tile* tiles, int w, int h, int sx, int sy, int sdir, int gx,
                                   int gy, int gdir) {
  if (!e || !tiles) return fail(PGTG_ERR_INVALID, "null argument");
  if (!e->cfg.fixed_map) return fail(PGTG_ERR_STATE, "config was not created with fixed_map");
  if (w != e->dc.W || h != e->dc.H) return fail(PGTG_ERR_INVALID, "fixed map size differs from the config");
  if (sx < 0 || sx >= w || sy < 0 || sy >= h || gx < 0 || gx >= w || gy < 0 || gy >= h || sdir < 0 || sdir > 3 || gdir < 0 || gdir > 3)
    return fail(PGTG_ERR_INVALID, "start/goal outside the map");
  std::vector<uint16_t> t((size_t)w * h);
  for (int i = 0; i < w * h; i++) {
    if (tiles[i].obstacle_type > 4 || tiles[i].obstacle_mask >= PGTG_NUM_MASKS) return fail(PGTG_ERR_INVALID, "bad obstacle type/mask");
    t[i] = (uint16_t)((tiles[i].exits & 15) | tiles[i].obstacle_type << 4 | (tiles[i].obstacle_type ? tiles[i].obstacle_mask : 0) << 7);
  }
  bk_set_device(e->device);
  uint16_t* d = dev_alloc<uint16_t>(e, t.size() + 1);
  if (!d) return fail(PGTG_ERR_CUDA, "device allocation failed");
  bk_h2d(d, t.data(), t.size() * 2, nullptr);
  bk_sync(nullptr);
  e->dp.fixed_tiles = d;
  e->dp.fixed_plan = plan_pack(sx, sy, sdir, gx, gy, gdir, 0);
  e->have_fixed = true;
  return PGTG_OK;
}

extern "C" int pgtg_load_direction_lut(pgtg_env* e, const uint8_t* lut, int radius) {
  if (!e || !lut) return fail(PGTG_ERR_INVALID, "null argument");
  if (radius != e->dc.lut_radius) return fail(PGTG_ERR_INVALID, "direction LUT radius must be max(width, height) in squares + 2");
  bk_set_device(e->device);
  size_t n = (size_t)(2 * radius + 1) * (2 * radius + 1);
  bk_h2d((void*)e->dp.dirlut, lut, n, nullptr);
  bk_sync(nullptr);
  return PGTG_OK;
}

extern "C" int pgtg_update_rules(pgtg_env* e, const pgtg_rule* rules, int num_rules) {
  if (!e || (num_rules > 0 && !rules)) return fail(PGTG_ERR_INVALID, "null argument");
  if (num_rules < 0 || num_rules > PGTG_MAX_RULES) return fail(PGTG_ERR_INVALID, "too many traffic rules");
  bk_set_device(e->device);
  bk_sync(nullptr);
  if (num_rules) bk_h2d((void*)e->dp.rules, rules, sizeof(pgtg_rule) * num_rules, nullptr);
  bk_sync(nullptr);
  e->dc.num_rules = num_rules;
  e->dc.rules_without_traffic = 0;
  for (int i = 0; i < num_rules; i++) if (rules[i].min_traffic <= 0 && rules[i].min_matching_traffic <= 0) e->dc.rules_without_traffic = 1;
  e->cfg.num_rules = num_rules;
  for (int i = 0; i < num_rules; i++) e->cfg.rules[i] = rules[i];
  // a rule that can fire without traffic needs apply_braking, which the lean tick does not contain
  e->dc.lean = e->cars_injected ? 0 : lean_predicate(e->cfg, e->dc);
  return PGTG_OK;
}

extern "C" int pgtg_load_draws(pgtg_env* e, const double* values, const uint8_t* tags, const int64_t* offsets) {
  if (!e || !offsets) return fail(PGTG_ERR_INVALID, "null argument");
  if (e->cfg.rng_mode != PGTG_RNG_TAPE) return fail(PGTG_ERR_STATE, "config was not created with rng_mode = PGTG_RNG_TAPE");
  size_t N = (size_t)e->dc.N;
  int64_t total = offsets[N];
  if (total < 0 || offsets[0] != 0) return fail(PGTG_ERR_INVALID, "bad tape offsets");
  bk_set_device(e->device);
  double* v = dev_alloc<double>(e, (size_t)total + 1, false);
  uint8_t* t = dev_alloc<uint8_t>(e, (size_t)total + 1, false);
  if (!v || !t) return fail(PGTG_ERR_CUDA, "device allocation failed");
  if (total) { bk_h2d(v, values, (size_t)total * 8, nullptr); bk_h2d(t, tags, (size_t)total, nullptr); }
  bk_h2d(e->dp.cursor, offsets, N * 8, nullptr);
  bk_h2d(e->dp.tape_end, offsets + 1, N * 8, nullptr);
  bk_sync(nullptr);
  e->dp.tape_values = v; e->dp.tape_tags = t;
  e->have_tape = true;
  return PGTG_OK;
}

static int join_side(pgtg_env* e, void* stream);
// One launch of the pregen pipeline (DESIGN.md 4.2). Launch L appends its map requests to queue L&1 and
// reads only ring slots filled by map generations <= L-2, so the map generation of launch L-1 (side
// stream, small persistent grid) runs concurrently with the tick of launch L. `join` makes the caller's
// stream wait for the generation just enqueued (full resets rewrite both ring slots).
static int run_pipeline(pgtg_env* e, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream, bool join) {
  if (!e->dc.pregen) {
    if (bk_launch(e, mode, mask, seeds, actions, action_bytes, stream)) return -1;
    e->launches++;
    return 0;
  }
  if (mode == MODE_STEP && inline_mapgen_now(e)) {  // no requests, no second kernel; maps of a reset may still be in flight
    if (join_side(e, stream)) return -1;
    const bool timed1 = e->timing && e->tev_used + 4 <= (int)e->tev.size();
    if (timed1) bk_event_record(e->tev[e->tev_used], stream);
    if (bk_launch(e, mode, mask, seeds, actions, action_bytes, stream)) return -1;
    e->launches++;
    if (timed1) { for (int i = 1; i < 4; i++) bk_event_record(e->tev[e->tev_used + i], stream); e->tev_used += 4; }
    e->launch_index++;
    return 0;
  }
  int par = (int)(e->launch_index & 1);
  e->dp.parity = par;
  // queue `par` was last read, and its ring slots last written, by the map generation of launch L-2
  if (e->launch_index >= 2 && bk_stream_wait(stream, e->ev_map[par])) return -1;
  if (bk_memset_async(e->dp.regen_count + par, 0, 4, stream)) return -1;
  bool timed = mode == MODE_STEP && e->timing && e->tev_used + 4 <= (int)e->tev.size();
  if (timed) bk_event_record(e->tev[e->tev_used], stream);
  if (bk_launch(e, mode, mask, seeds, actions, action_bytes, stream)) return -1;
  e->launches++;
  if (timed) bk_event_record(e->tev[e->tev_used + 1], stream);
  void* ms = e->overlap ? e->side_stream : stream;  // overlap off: the generation follows the tick on the caller's stream
  if (e->overlap && (bk_event_record(e->ev_tick, stream) || bk_stream_wait(e->side_stream, e->ev_tick))) return -1;
  if (timed) bk_event_record(e->tev[e->tev_used + 2], ms);
  if (bk_launch(e, MODE_MAPGEN, nullptr, nullptr, nullptr, 0, ms)) return -1;
  e->launches++;
  if (timed) { bk_event_record(e->tev[e->tev_used + 3], ms); e->tev_used += 4; }
  if (bk_event_record(e->ev_map[par], ms)) return -1;
  if (join && bk_stream_wait(stream, e->ev_map[par])) return -1;
  e->launch_index++;
  return 0;
}

// make `stream` wait for every map generation in flight (before resets, host reads and timing joins)
static int join_side(pgtg_env* e, void* stream) {
  if (!e->dc.pregen || e->launch_index == 0) return 0;
  if (bk_stream_wait(stream, e->ev_map[0])) return -1;
  if (e->launch_index >= 2 && bk_stream_wait(stream, e->ev_map[1])) return -1;
  return 0;
}

static int check_ready(pgtg_env* e) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  if (e->cfg.fixed_map && !e->have_fixed) return fail(PGTG_ERR_STATE, "fixed_map config: call pgtg_load_fixed_map first");
  if (e->cfg.rng_mode == PGTG_RNG_TAPE && !e->have_tape) return fail(PGTG_ERR_STATE, "conformance mode: call pgtg_load_draws first");
  return PGTG_OK;
}

extern "C" int pgtg_reset(pgtg_env* e, const int64_t* seeds, const uint8_t* mask, void* stream) {
  int rc = check_ready(e);
  if (rc) return rc;
  bk_set_device(e->device);
  size_t N = (size_t)e->dc.N;
  if (!e->did_reset && mask) return fail(PGTG_ERR_STATE, "the first reset must cover all envs");
  if (seeds) bk_h2d(e->seeds_dev, seeds, N * 8, stream);
  if (mask) bk_h2d(e->mask_dev, mask, N, stream);
  // a reset rewrites both ring slots of the envs it touches: let every map generation in flight finish first
  if (join_side(e, stream)) return fail(PGTG_ERR_CUDA, std::string("stream wait failed: ") + bk_error());
  if (run_pipeline(e, MODE_RESET, mask ? e->mask_dev : nullptr, seeds ? e->seeds_dev : nullptr, nullptr, 0, stream, true))
    return fail(PGTG_ERR_CUDA, std::string("reset launch failed: ") + bk_error());
  e->did_reset = true;
  return PGTG_OK;
}

extern "C" int pgtg_step(pgtg_env* e, const void* actions_dev, int action_bytes, void* stream) {
  int rc = check_ready(e);
  if (rc) return rc;
  if (!e->did_reset) return fail(PGTG_ERR_STATE, "step before reset");
  if (!actions_dev || (action_bytes != 4 && action_bytes != 8)) return fail(PGTG_ERR_INVALID, "actions must be device int32 or int64");
  bk_set_device(e->device);
  if (e->dc.pregen) {
    if (run_pipeline(e, MODE_STEP, nullptr, nullptr, actions_dev, action_bytes, stream, false))
      return fail(PGTG_ERR_CUDA, std::string("step launch failed: ") + bk_error());
  } else {
    bool timed = e->timing && e->tev_used + 4 <= (int)e->tev.size();
    if (timed) bk_event_record(e->tev[e->tev_used], stream);
    if (bk_launch(e, MODE_STEP, nullptr, nullptr, actions_dev, action_bytes, stream))
      return fail(PGTG_ERR_CUDA, std::string("step launch failed: ") + bk_error());
    e->launches++;
    if (timed) { for (int k = 1; k < 4; k++) bk_event_record(e->tev[e->tev_used + k], stream); e->tev_used += 4; }
  }
  return PGTG_OK;
}

extern "C" int pgtg_step_host(pgtg_env* e, const int32_t* actions, int8_t* obs_map, int32_t* obs_position,
                              int32_t* obs_velocity, double* reward, uint8_t* terminated, uint8_t* truncated, void* stream) {
  if (!e || !actions) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  size_t N = (size_t)e->dc.N;
  bk_h2d(e->actions_dev, actions, N * 4, stream);
  int rc = pgtg_step(e, e->actions_dev, 4, stream);
  if (rc) return rc;
  if (obs_map) bk_d2h(obs_map, e->dp.obs_map, N * e->dc.obs_bits, stream);
  if (obs_position) bk_d2h(obs_position, e->dp.obs_position, N * 8, stream);
  if (obs_velocity) bk_d2h(obs_velocity, e->dp.obs_velocity, N * 8, stream);
  if (reward) bk_d2h(reward, e->dp.reward, N * 8, stream);
  if (terminated) bk_d2h(terminated, e->dp.terminated, N, stream);
  if (truncated) bk_d2h(truncated, e->dp.truncated, N, stream);
  if (bk_sync(stream)) return fail(PGTG_ERR_CUDA, std::string("step failed: ") + bk_error());
  return PGTG_OK;
}

extern "C" int pgtg_get_buffers(pgtg_env* e, pgtg_buffers* out) {
  if (!e || !out) return fail(PGTG_ERR_INVALID, "null argument");
  memset(out, 0, sizeof *out);
  const DevPtrs& p = e->dp;
  out->num_envs = e->dc.N; out->num_channels = e->dc.C; out->window = e->dc.P; out->max_cars = e->dc.max_cars;
  out->obs_map = p.obs_map; out->obs_position = p.obs_position; out->obs_velocity = p.obs_velocity;
  out->obs_next_subgoal_direction = p.obs_nsd; out->reward = p.reward; out->cost = p.cost;
  out->terminated = p.terminated; out->truncated = p.truncated; out->step_state = p.step_state; out->step_flags = p.step_flags;
  out->final_obs_map = p.f_obs_map; out->final_obs_position = p.f_obs_position; out->final_obs_velocity = p.f_obs_velocity;
  out->final_obs_next_subgoal_direction = p.f_obs_nsd; out->stats = p.stats;
  return PGTG_OK;
}

// ---- DLPack (v0 ABI) ---------------------------------------------------------------------------
struct DLDevice_ { int32_t device_type; int32_t device_id; };
struct DLDataType_ { uint8_t code; uint8_t bits; uint16_t lanes; };
struct DLTensor_ { void* data; DLDevice_ device; int32_t ndim; DLDataType_ dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset; };
struct DLManagedTensor_ { DLTensor_ dl_tensor; void* manager_ctx; void (*deleter)(DLManagedTensor_*); };
struct DLHolder { DLManagedTensor_ mt; int64_t shape[4]; };
static void dl_deleter(DLManagedTensor_* mt) { delete (DLHolder*)mt->manager_ctx; }

extern "C" int pgtg_dlpack(pgtg_env* e, const char* name, void** out) {
  if (!e || !name || !out) return fail(PGTG_ERR_INVALID, "null argument");
  const DevCfg& c = e->dc;
  const DevPtrs& p = e->dp;
  struct Spec { const char* name; void* ptr; int code, bits, ndim; int64_t shape[4]; };
  int64_t N = c.N, C = c.C, P = c.P;
  const Spec specs[] = {
      {"obs_map", p.obs_map, 0, 8, 4, {N, C, P, P}},
      {"obs_position", p.obs_position, 0, 32, 2, {N, 2}},
      {"obs_velocity", p.obs_velocity, 0, 32, 2, {N, 2}},
      {"obs_next_subgoal_direction", p.obs_nsd, 0, 32, 1, {N}},
      {"reward", p.reward, 2, 64, 1, {N}},
      {"cost", p.cost, 2, 64, 1, {N}},
      {"terminated", p.terminated, 1, 8, 1, {N}},
      {"truncated", p.truncated, 1, 8, 1, {N}},
      {"step_state", p.step_state, 0, 32, 2, {N, 4}},
      {"step_flags", p.step_flags, 1, 8, 1, {N}},
      {"final_obs_map", p.f_obs_map, 0, 8, 4, {N, C, P, P}},
      {"final_obs_position", p.f_obs_position, 0, 32, 2, {N, 2}},
      {"final_obs_velocity", p.f_obs_velocity, 0, 32, 2, {N, 2}},
      {"final_obs_next_subgoal_direction", p.f_obs_nsd, 0, 32, 1, {N}},
      {"stats", p.stats, 2, 64, 1, {8}},
      {"obs_flat", e->flat, 2, 32, 2, {N, (int64_t)e->flat_dim}},
  };
  for (const Spec& s : specs) {
    if (strcmp(s.name, name)) continue;
    if (!s.ptr) return fail(PGTG_ERR_STATE, std::string("buffer not allocated in this configuration: ") + name);
    DLHolder* h = new DLHolder();
    for (int i = 0; i < s.ndim; i++) h->shape[i] = s.shape[i];
    h->mt.dl_tensor.data = s.ptr;
    h->mt.dl_tensor.device.device_type = bk_dl_device_type();
    h->mt.dl_tensor.device.device_id = e->device;
    h->mt.dl_tensor.ndim = s.ndim;
    h->mt.dl_tensor.dtype.code = (uint8_t)s.code; h->mt.dl_tensor.dtype.bits = (uint8_t)s.bits; h->mt.dl_tensor.dtype.lanes = 1;
    h->mt.dl_tensor.shape = h->shape; h->mt.dl_tensor.strides = nullptr; h->mt.dl_tensor.byte_offset = 0;
    h->mt.manager_ctx = h; h->mt.deleter = dl_deleter;
    *out = &h->mt;
    return PGTG_OK;
  }
  return fail(PGTG_ERR_INVALID, std::string("unknown buffer name: ") + name);
}

extern "C" int pgtg_get_state(pgtg_env* e, pgtg_state* s) {
  if (!e || !s) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  const DevCfg& c = e->dc;
  const DevPtrs& p = e->dp;
  size_t N = (size_t)c.N;
  std::vector<short4> agent(N);
  std::vector<uint32_t> misc(N), tmp(N);
  bk_d2h(agent.data(), p.agent, N * sizeof(short4), nullptr);
  bk_d2h(misc.data(), p.misc, N * 4, nullptr);
  bk_sync(nullptr);
  for (size_t i = 0; i < N; i++) {
    if (s->agent) { s->agent[4 * i] = agent[i].x; s->agent[4 * i + 1] = agent[i].y; s->agent[4 * i + 2] = agent[i].z; s->agent[4 * i + 3] = agent[i].w; }
    if (s->flat_tire) s->flat_tire[i] = (uint8_t)(misc[i] & 1);
    if (s->light_counter) s->light_counter[i] = (int32_t)misc_light(misc[i]);
    if (s->num_cars) s->num_cars[i] = (int32_t)(misc[i] >> 16);
  }
  if (s->elapsed) { bk_d2h(tmp.data(), p.elapsed, N * 4, nullptr); bk_sync(nullptr); for (size_t i = 0; i < N; i++) s->elapsed[i] = (int32_t)tmp[i]; }
  if (s->cars) {
    size_t MC = (size_t)c.max_cars;
    std::vector<uint64_t> cars(2 * MC * N);
    bk_d2h(cars.data(), p.cars, 2 * MC * N * 8, nullptr);
    bk_sync(nullptr);
    memset(s->cars, 0, sizeof(int32_t) * N * MC * 7);
    for (size_t i = 0; i < N; i++) {
      size_t n = misc[i] >> 16;
      const uint64_t* live = cars.data() + (2 * i + misc_half(misc[i])) * MC;
      for (size_t k = 0; k < n && k < MC; k++) {
        Car car = car_unpack(live[k]);
        int32_t* o = s->cars + (i * MC + k) * 7;
        o[0] = (int32_t)car.id; o[1] = car.x; o[2] = car.y; o[3] = car.route; o[4] = car.profile; o[5] = car.patience; o[6] = car.delay;
      }
    }
  }
  if (s->tiles || s->used) {
    std::vector<uint16_t> tiles(N * c.T);
    bk_d2h(tiles.data(), p.tiles, N * c.T * 2, nullptr);
    bk_sync(nullptr);
    for (size_t i = 0; i < N * (size_t)c.T; i++) {
      if (s->tiles) s->tiles[i] = (uint16_t)(tiles[i] & 0x3FFF);
      if (s->used) s->used[i] = (uint8_t)((tiles[i] >> 14) & 1);
    }
  }
  if (s->plan) {
    bk_d2h(tmp.data(), p.plan, N * 4, nullptr);
    bk_sync(nullptr);
    for (size_t i = 0; i < N; i++) {
      int32_t* o = s->plan + 8 * i;
      unsigned pl = tmp[i];
      o[0] = plan_sx(pl); o[1] = plan_sy(pl); o[2] = plan_sd(pl); o[3] = plan_gx(pl); o[4] = plan_gy(pl); o[5] = plan_gd(pl); o[6] = plan_ns(pl); o[7] = 0;
    }
  }
  if (s->draw_cursor) {
    if (p.cursor) { bk_d2h(s->draw_cursor, p.cursor, N * 8, nullptr); bk_sync(nullptr); }
    else memset(s->draw_cursor, 0, N * 8);
  }
  if (s->error) { bk_d2h(s->error, p.error, N * 4, nullptr); bk_sync(nullptr); }
  return PGTG_OK;
}

extern "C" int pgtg_set_state(pgtg_env* e, const pgtg_state* s) {
  // set_to_state (environment.py:1301-1342): position, velocity, flat_tire and cars only
  if (!e || !s) return fail(PGTG_ERR_INVALID, "null argument");
  if (!e->did_reset) return fail(PGTG_ERR_STATE, "set_state before reset");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  const DevCfg& c = e->dc;
  const DevPtrs& p = e->dp;
  size_t N = (size_t)c.N, MC = (size_t)c.max_cars;
  if (s->agent) {
    std::vector<short4> agent(N);
    for (size_t i = 0; i < N; i++) { agent[i].x = (short)s->agent[4 * i]; agent[i].y = (short)s->agent[4 * i + 1]; agent[i].z = (short)s->agent[4 * i + 2]; agent[i].w = (short)s->agent[4 * i + 3]; }
    bk_h2d(p.agent, agent.data(), N * sizeof(short4), nullptr);
  }
  std::vector<uint32_t> misc(N);
  bk_d2h(misc.data(), p.misc, N * 4, nullptr);
  bk_sync(nullptr);
  if (s->flat_tire) for (size_t i = 0; i < N; i++) misc[i] = (misc[i] & ~1u) | (s->flat_tire[i] ? 1u : 0u);
  if (s->cars && s->num_cars) {
    std::vector<uint64_t> cars(2 * MC * N, 0);
    std::vector<uint32_t> next_id(N);
    bk_d2h(next_id.data(), p.next_car_id, N * 4, nullptr);
    bk_sync(nullptr);
    for (size_t i = 0; i < N; i++) {
      size_t n = (size_t)s->num_cars[i];
      if (n > MC) return fail(PGTG_ERR_INVALID, "more cars than max_cars");
      for (size_t k = 0; k < n; k++) {
        const int32_t* o = s->cars + (i * MC + k) * 7;
        Car car; car.id = (unsigned)o[0]; car.x = o[1]; car.y = o[2]; car.route = o[3]; car.profile = o[4]; car.patience = 0; car.delay = 0;
        cars[(2 * i + misc_half(misc[i])) * MC + k] = car_pack(car);
        if (k == n - 1) next_id[i] = (unsigned)o[0] + 1;  // :1340
      }
      misc[i] = (misc[i] & 0xFFFFu) | (uint32_t)n << 16;
      if (n > 0) { e->cars_injected = true; e->dc.lean = 0; }  // cars injected into a no-traffic handle: from now on the general tick
    }
    bk_h2d(p.cars, cars.data(), 2 * MC * N * 8, nullptr);
    bk_h2d(p.next_car_id, next_id.data(), N * 4, nullptr);
  }
  bk_h2d(p.misc, misc.data(), N * 4, nullptr);
  bk_sync(nullptr);
  return PGTG_OK;
}

extern "C" int pgtg_get_info(pgtg_env* e, int32_t* agent_direction, int32_t* current_tile_type, int32_t* profile_counts) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  if (!e->did_reset) return fail(PGTG_ERR_STATE, "get_info before reset");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  const size_t N = (size_t)e->dc.N;
  if (!e->info_dev && !(e->info_dev = dev_alloc<int32_t>(e, 7 * N))) return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error());
  if (bk_info(e, e->info_dev)) return fail(PGTG_ERR_CUDA, std::string("info launch failed: ") + bk_error());
  e->launches++;
  if (agent_direction) bk_d2h(agent_direction, e->info_dev, N * 4, nullptr);
  if (current_tile_type) bk_d2h(current_tile_type, e->info_dev + N, N * 4, nullptr);
  if (profile_counts) {  // device layout [5][N] -> caller layout [N][5]
    std::vector<int32_t> tmp(5 * N);
    bk_d2h(tmp.data(), e->info_dev + 2 * N, 5 * N * 4, nullptr);
    bk_sync(nullptr);
    for (size_t i = 0; i < N; i++) for (int q = 0; q < 5; q++) profile_counts[i * 5 + q] = tmp[(size_t)q * N + i];
  }
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  return PGTG_OK;
}


// ---- full-state checkpoint / clone (PGTGEnv.light_step deep-copies the env, environment.py:1283-1299) ------------
// Everything a tick reads or writes: SoA state, both ring slots and the map-request queues, car lists, RNG state
// (numpy mode) / tape cursors, episode statistics, the output buffers, plus the host-side pipeline position.
struct StateHeader { uint64_t magic, total_bytes, launch_index; int32_t parity, did_reset, cars_injected, lean, n_allocs, reserved; };
static const uint64_t STATE_MAGIC = 0x5047544753544132ull;  // "PGTGSTA2"
static size_t state_payload_bytes(const pgtg_env* e) { size_t n = 0; for (auto& s : e->state_allocs) n += (s.bytes + 15) & ~(size_t)15; return n; }

extern "C" int64_t pgtg_state_bytes(pgtg_env* e) { return e ? (int64_t)(sizeof(StateHeader) + state_payload_bytes(e)) : 0; }

extern "C" int pgtg_save_state(pgtg_env* e, void* out, int64_t out_bytes) {
  if (!e || !out) return fail(PGTG_ERR_INVALID, "null argument");
  if (out_bytes < pgtg_state_bytes(e)) return fail(PGTG_ERR_INVALID, "state buffer too small (see pgtg_state_bytes)");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  StateHeader h = {STATE_MAGIC, (uint64_t)pgtg_state_bytes(e), e->launch_index, e->dp.parity, e->did_reset, e->cars_injected, e->dc.lean, (int32_t)e->state_allocs.size(), 0};
  memcpy(out, &h, sizeof h);
  unsigned char* dst = (unsigned char*)out + sizeof h;
  for (auto& s : e->state_allocs) { bk_d2h(dst, s.ptr, s.bytes, nullptr); dst += (s.bytes + 15) & ~(size_t)15; }
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  return PGTG_OK;
}

extern "C" int pgtg_load_state(pgtg_env* e, const void* in, int64_t in_bytes) {
  if (!e || !in) return fail(PGTG_ERR_INVALID, "null argument");
  StateHeader h;
  if (in_bytes < (int64_t)sizeof h) return fail(PGTG_ERR_INVALID, "not a pgtg state blob");
  memcpy(&h, in, sizeof h);
  if (h.magic != STATE_MAGIC || (int64_t)h.total_bytes != pgtg_state_bytes(e) || in_bytes < (int64_t)h.total_bytes || h.n_allocs != (int32_t)e->state_allocs.size())
    return fail(PGTG_ERR_INVALID, "state blob does not belong to a handle of this configuration");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  const unsigned char* src = (const unsigned char*)in + sizeof h;
  for (auto& s : e->state_allocs) { bk_h2d(s.ptr, src, s.bytes, nullptr); src += (s.bytes + 15) & ~(size_t)15; }
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  e->launch_index = h.launch_index; e->dp.parity = h.parity; e->did_reset = h.did_reset != 0; e->cars_injected = h.cars_injected != 0; e->dc.lean = h.lean;
  return PGTG_OK;
}

// device-to-device: dst becomes an exact copy of src (same configuration, same device)
extern "C" int pgtg_copy_state(pgtg_env* dst, pgtg_env* src) {
  if (!dst || !src) return fail(PGTG_ERR_INVALID, "null argument");
  if (dst->device != src->device || dst->state_allocs.size() != src->state_allocs.size()) return fail(PGTG_ERR_INVALID, "handles differ in configuration or device");
  for (size_t i = 0; i < src->state_allocs.size(); i++)
    if (dst->state_allocs[i].bytes != src->state_allocs[i].bytes) return fail(PGTG_ERR_INVALID, "handles differ in configuration");
  bk_set_device(src->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  for (size_t i = 0; i < src->state_allocs.size(); i++) bk_d2d(dst->state_allocs[i].ptr, src->state_allocs[i].ptr, src->state_allocs[i].bytes, nullptr);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  dst->launch_index = src->launch_index; dst->dp.parity = src->dp.parity; dst->did_reset = src->did_reset; dst->cars_injected = src->cars_injected;
  dst->dc.lean = src->dc.lean; dst->dc.num_rules = src->dc.num_rules; dst->dc.rules_without_traffic = src->dc.rules_without_traffic;
  dst->dc.max_episode_steps = src->dc.max_episode_steps;
  return PGTG_OK;
}

// ---- evaluator statistics (ModularEvaluator.evaluate, evaluator.py:292-339) ----------------------------------------
// gamma > 0 switches on the per-env discounted return total += reward * pow(gamma, t) (t = tick of the episode) and the
// two statistics built on it: stats[6] = sum of the discounted returns of finished episodes, stats[7] = how many of them
// were negative. max_steps becomes the episode cap (the evaluator's "over max_steps" = truncations, stats[5]).
extern "C" int pgtg_set_evaluation(pgtg_env* e, double gamma, int max_steps) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  if (!(gamma > 0)) { e->dc.eval_on = 0; return PGTG_OK; }
  if (max_steps < 1) return fail(PGTG_ERR_INVALID, "max_steps must be >= 1");
  std::vector<double> tab((size_t)max_steps);
  for (int t = 0; t < max_steps; t++) tab[(size_t)t] = pow(gamma, (double)t);  // np.power(GAMMA, t) calls the same libm pow
  double* td = dev_alloc<double>(e, (size_t)max_steps, false);
  if (!td) return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error());
  bk_h2d(td, tab.data(), tab.size() * 8, nullptr);
  if (!e->dp.ep_disc) {
    e->dp.ep_disc = dev_alloc<double>(e, (size_t)e->dc.N);
    if (!e->dp.ep_disc) return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error());
    e->state_allocs.push_back({e->dp.ep_disc, 8 * (size_t)e->dc.N});
  } else bk_memset(e->dp.ep_disc, 0, 8 * (size_t)e->dc.N);
  bk_sync(nullptr);
  e->dp.gamma_pow = td;
  e->dc.eval_on = 1; e->dc.gamma_len = max_steps; e->dc.max_episode_steps = max_steps; e->cfg.max_episode_steps = max_steps;
  return PGTG_OK;
}

// ---- host-buffer step with the observation planes as bits, double-buffered ------------------------------------------
// H2D actions -> tick -> one device-to-device gather of the step's outputs into staging slot (k & 1) -> D2H of that slot on
// a copy stream. The tick of call k + 1 does not wait for the copies of call k (it only needs slot (k + 1) & 1, whose
// copies belong to call k - 1). wait != 0: return when this call's outputs are in the host buffers; wait == 0: they are
// complete after the next pgtg_host_sync (or the next call with the same slot parity).
struct HostLayout { size_t packed, pos, vel, reward, term, trunc, total; };
static HostLayout host_layout(const pgtg_env* e) {
  HostLayout L; size_t N = (size_t)e->dc.N, o = 0;
  auto take = [&](size_t b) { size_t at = o; o += (b + 255) & ~(size_t)255; return at; };
  L.packed = take(4 * ((N * e->dc.obs_bits + 31) / 32)); L.pos = take(8 * N); L.vel = take(8 * N); L.reward = take(8 * N); L.term = take(N); L.trunc = take(N);
  L.total = o;
  return L;
}
extern "C" int64_t pgtg_packed_obs_bytes(pgtg_env* e) { return e ? (int64_t)(4 * (((size_t)e->dc.N * e->dc.obs_bits + 31) / 32)) : 0; }

extern "C" int pgtg_step_host_packed(pgtg_env* e, const int32_t* actions, uint32_t* obs_packed, int32_t* obs_position, int32_t* obs_velocity,
                                     double* reward, uint8_t* terminated, uint8_t* truncated, int wait, void* stream) {
  if (!e || !actions) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  const size_t N = (size_t)e->dc.N;
  const HostLayout L = host_layout(e);
  if (!e->packed_dev) {
    e->packed_dev = dev_alloc<uint32_t>(e, (size_t)pgtg_packed_obs_bytes(e) / 4 + 8);
    e->stage_dev[0] = dev_alloc<unsigned char>(e, L.total); e->stage_dev[1] = dev_alloc<unsigned char>(e, L.total);
    e->copy_stream = bk_stream_create();
    for (int i = 0; i < 2; i++) { e->ev_stage[i] = bk_event_create(); e->ev_copied[i] = bk_event_create(); }
    if (!e->packed_dev || !e->stage_dev[0] || !e->stage_dev[1] || !e->copy_stream || !e->ev_copied[1]) return fail(PGTG_ERR_CUDA, std::string("allocation failed: ") + bk_error());
    e->stage_bytes = L.total;
    e->dp.obs_packed = e->packed_dev;  // from now on the ticks also store the planes as bits
  }
  const int slot = (int)(e->host_steps & 1);
  bk_h2d(e->actions_dev, actions, N * 4, stream);
  int rc = pgtg_step(e, e->actions_dev, 4, stream);
  if (rc) return rc;
  // slot's previous copies (call k - 2) must have left the staging buffer
  if (e->host_steps >= 2 && bk_stream_wait(stream, e->ev_copied[slot])) return fail(PGTG_ERR_CUDA, std::string("stream wait failed: ") + bk_error());
  unsigned char* st = e->stage_dev[slot];
  bk_d2d(st + L.packed, e->dp.obs_packed, (size_t)pgtg_packed_obs_bytes(e), stream);
  bk_d2d(st + L.pos, e->dp.obs_position, 8 * N, stream); bk_d2d(st + L.vel, e->dp.obs_velocity, 8 * N, stream);
  bk_d2d(st + L.reward, e->dp.reward, 8 * N, stream); bk_d2d(st + L.term, e->dp.terminated, N, stream); bk_d2d(st + L.trunc, e->dp.truncated, N, stream);
  if (bk_event_record(e->ev_stage[slot], stream) || bk_stream_wait(e->copy_stream, e->ev_stage[slot])) return fail(PGTG_ERR_CUDA, std::string("event failed: ") + bk_error());
  void* cs = e->copy_stream;
  if (obs_packed) bk_d2h(obs_packed, st + L.packed, (size_t)pgtg_packed_obs_bytes(e), cs);
  if (obs_position) bk_d2h(obs_position, st + L.pos, 8 * N, cs);
  if (obs_velocity) bk_d2h(obs_velocity, st + L.vel, 8 * N, cs);
  if (reward) bk_d2h(reward, st + L.reward, 8 * N, cs);
  if (terminated) bk_d2h(terminated, st + L.term, N, cs);
  if (truncated) bk_d2h(truncated, st + L.trunc, N, cs);
  if (bk_event_record(e->ev_copied[slot], cs)) return fail(PGTG_ERR_CUDA, std::string("event failed: ") + bk_error());
  e->host_steps++;
  if (wait && bk_sync(cs)) return fail(PGTG_ERR_CUDA, std::string("step failed: ") + bk_error());
  return PGTG_OK;
}

// wait for every copy of the host-buffer steps issued so far
extern "C" int pgtg_host_sync(pgtg_env* e) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  if (e->copy_stream && bk_sync(e->copy_stream)) return fail(PGTG_ERR_CUDA, std::string("copy failed: ") + bk_error());
  return PGTG_OK;
}

// bits -> int8 cells on the host (callers that want the [N, C, P, P] planes back), `threads` worker threads
#include <thread>
extern "C" int pgtg_unpack_obs(const uint32_t* packed, int8_t* obs_map, int64_t n_cells, int threads) {
  if (!packed || !obs_map || n_cells < 0) return fail(PGTG_ERR_INVALID, "null argument");
  if (threads < 1) threads = 1;
  auto work = [&](int64_t lo, int64_t hi) {  // [lo, hi) in units of 32 cells
    for (int64_t w = lo; w < hi; w++) {
      const uint32_t v = packed[w];
      uint64_t* out = (uint64_t*)(obs_map + 32 * w);
      for (int b = 0; b < 4; b++) {  // 8 bits -> 8 bytes: replicate the byte, keep bit k in byte k, normalise to 0 / 1
        const uint64_t x = (v >> (8 * b)) & 255u;
        out[b] = ((((x * 0x0101010101010101ull) & 0x8040201008040201ull) + 0x7F7F7F7F7F7F7F7Full) >> 7) & 0x0101010101010101ull;
      }
    }
  };
  const int64_t words = n_cells / 32;
  std::vector<std::thread> pool;
  for (int t = 0; t < threads; t++) pool.emplace_back(work, words * t / threads, words * (t + 1) / threads);
  for (auto& th : pool) th.join();
  for (int64_t i = words * 32; i < n_cells; i++) obs_map[i] = (int8_t)((packed[i >> 5] >> (i & 31)) & 1u);
  return PGTG_OK;
}

extern "C" int pgtg_reduce_stats(pgtg_env* e, void* stream) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  if (join_side(e, stream)) return fail(PGTG_ERR_CUDA, std::string("stream wait failed: ") + bk_error());
  if (bk_stats_reduce(e, stream)) return fail(PGTG_ERR_CUDA, std::string("stats reduction failed: ") + bk_error());
  return PGTG_OK;
}

extern "C" int pgtg_reset_stats(pgtg_env* e, void* stream) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  if (bk_stats_reset(e, stream)) return fail(PGTG_ERR_CUDA, std::string("stats reset failed: ") + bk_error());
  return PGTG_OK;
}

extern "C" int pgtg_stats(pgtg_env* e, double* out8, int reset_after) {
  if (!e || !out8) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  // ticks may be in flight on non-blocking streams: the reduction below runs on the legacy stream
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  if (bk_stats_reduce(e, nullptr)) return fail(PGTG_ERR_CUDA, std::string("stats reduction failed: ") + bk_error());
  bk_d2h(out8, e->dp.stats, 64, nullptr);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  if (reset_after) { bk_stats_reset(e, nullptr); bk_sync(nullptr); }
  return PGTG_OK;
}

// Flattened observation, float32 [N, D], in the order of gymnasium 0.28.1 `FlattenObservation` over the
// reference's Dict space (train.py:39-40): Dict keys sorted -> "map" (sub-keys sorted, each plane
// P*P cells, index [x][y]), "next_subgoal_direction" (one-hot 9, value + 1), "position" (two one-hots
// of 9), "velocity" (2). `plane_order[i]` = channel index of the i-th plane in sorted-key order.
extern "C" int pgtg_flatten(pgtg_env* e, const int32_t* plane_order, void* stream, float** out_dev, int* out_dim) {
  if (!e || !plane_order) return fail(PGTG_ERR_INVALID, "null argument");
  if (!e->did_reset) return fail(PGTG_ERR_STATE, "flatten before reset");
  bk_set_device(e->device);
  const DevCfg& c = e->dc;
  int dim = c.C * c.P * c.P + (c.use_nsd ? 9 : 0) + 18 + 2;
  if (!e->flat) {
    e->flat = dev_alloc<float>(e, (size_t)c.N * dim, false);
    if (!e->flat) return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error());
    e->flat_dim = dim;
  }
  for (int i = 0; i < c.C; i++) {
    if (plane_order[i] < 0 || plane_order[i] >= c.C) return fail(PGTG_ERR_INVALID, "bad plane order");
    e->flat_order[i] = plane_order[i];
  }
  if (bk_flatten(e, stream)) return fail(PGTG_ERR_CUDA, std::string("flatten launch failed: ") + bk_error());
  e->launches++;
  if (out_dev) *out_dev = e->flat;
  if (out_dim) *out_dim = dim;
  return PGTG_OK;
}

// OR of every env's sticky error flags (1 tape overrun, 2 tape tag mismatch, 4 tape index out of range, 8 goal unreachable,
// 16 no route at a spawn square, 32 more cars than max_cars, 64 no start square, 128 action outside 0..8). Synchronises.
extern "C" int pgtg_error_summary(pgtg_env* e, uint32_t* out_flags) {
  if (!e || !out_flags) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  if (!e->info_dev && !(e->info_dev = dev_alloc<int32_t>(e, 7 * (size_t)e->dc.N))) return fail(PGTG_ERR_CUDA, std::string("device allocation failed: ") + bk_error());
  if (bk_error_or(e, (uint32_t*)e->info_dev)) return fail(PGTG_ERR_CUDA, std::string("launch failed: ") + bk_error());
  e->launches++;
  bk_d2h(out_flags, e->info_dev, 4, nullptr);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  return PGTG_OK;
}

extern "C" int64_t pgtg_launch_count(pgtg_env* e) { return e ? e->launches : 0; }

// Which kernels a step of this handle launches, as text (bench / test reports).
extern "C" int pgtg_kernel_info(pgtg_env* e, char* out, int out_bytes) {
  if (!e || !out || out_bytes < 1) return fail(PGTG_ERR_INVALID, "null argument");
  const char* rng = e->cfg.rng_mode == PGTG_RNG_TAPE ? "tape" : e->cfg.rng_mode == PGTG_RNG_NUMPY ? "numpy" : "philox";
  if (e->traffic_G > 0) snprintf(out, (size_t)out_bytes, "tick=traffic(G=%d,NT=%d) mapgen=%s rng=%s", e->traffic_G, e->traffic_NT, e->dc.pregen ? (e->dc.conn_bits && e->dc.path_tab ? "tabled" : "general") : "none", rng);
  else snprintf(out, (size_t)out_bytes, "tick=%s(B=%d) mapgen=%s rng=%s", e->dc.lean && e->dc.pregen && e->cfg.rng_mode != PGTG_RNG_TAPE && !getenv("PGTG_NO_LEAN") ? (e->dc.lean == 2 ? (e->dc.write_final_obs ? "lean+slide+final" : "lean+slide") : e->dc.write_final_obs ? "lean+final" : "lean") : "general", e->block,
                e->dc.pregen ? (e->dc.conn_bits && e->dc.path_tab ? "tabled" : "general") : "in-tick", rng);
  return PGTG_OK;
}

// Per-kernel device timing: while enabled, pgtg_step brackets each of its kernels with CUDA events on
// the launching stream (up to max_steps ticks). pgtg_timing synchronises and returns the summed
// durations (ms) of the tick kernel and of the map-generation kernel over the recorded ticks.
extern "C" int pgtg_enable_timing(pgtg_env* e, int max_steps) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  e->timing = max_steps > 0;
  e->tev_used = 0;
  while ((int)e->tev.size() < 4 * max_steps) {
    void* ev = bk_event_create();
    if (!ev) return fail(PGTG_ERR_CUDA, std::string("event creation failed: ") + bk_error());
    e->tev.push_back(ev);
  }
  return PGTG_OK;
}

// Overlap of map generation with the next tick (default on). Off = the two kernels run back to back on
// the caller's stream with a full-size generation grid: used to time each kernel alone.
extern "C" int pgtg_set_overlap(pgtg_env* e, int on) {
  if (!e) return fail(PGTG_ERR_INVALID, "null handle");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  e->overlap = on != 0;
  e->mapgen_grid = on ? e->mapgen_grid_overlap : 0;
  return PGTG_OK;
}

extern "C" int pgtg_timing(pgtg_env* e, double* tick_ms, double* mapgen_ms, int* steps) {
  if (!e || !tick_ms || !mapgen_ms || !steps) return fail(PGTG_ERR_INVALID, "null argument");
  bk_set_device(e->device);
  if (bk_sync(nullptr)) return fail(PGTG_ERR_CUDA, std::string("device error: ") + bk_error());
  *tick_ms = *mapgen_ms = 0;
  *steps = e->tev_used / 4;
  for (int i = 0; i + 3 < e->tev_used; i += 4) {  // [tick begin, tick end] on the caller's stream, [mapgen begin, end] on the side stream
    *tick_ms += bk_event_elapsed(e->tev[i], e->tev[i + 1]);
    *mapgen_ms += bk_event_elapsed(e->tev[i + 2], e->tev[i + 3]);
  }
  e->tev_used = 0;
  return PGTG_OK;
}
