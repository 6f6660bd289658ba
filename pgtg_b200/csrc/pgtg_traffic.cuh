// pgtg_traffic.cuh -- the traffic tick: phases of the kernel that runs every configuration with cars
// (Philox mode). Compiled by nvcc into pgtg_traffic.cu and by g++ into tests/emu (phases as loops).
//
// The sequential tick (one env per thread, cars in a loop) cannot fill a B200: 10 of 32 lanes active,
// one wave of warps, every car drawing Philox words inside a divergent loop. Here a CTA owns G envs and
// switches between two mappings, phase by phase, through shared memory:
//
//   flat over cars   every thread takes one (env, car) item of the CTA's G car lists: the per-car work
//                    that does not depend on other cars -- Philox block, move gating, probe of the four
//                    neighbour squares in the lane tables, traffic-light decision, push-through draw,
//                    respawn square / profile / route -- becomes an INTENT word; later the commit of the
//                    resolved list, the creation of a new episode's cars, and the traffic plane;
//   one env/thread   what the reference defines sequentially: blocking in list order (a car sees the cars
//                    before it at their new squares and the ones after it at their old squares,
//                    environment.py:944-962, 1121-1127), then the agent's move, reward, termination,
//                    auto-reset and the map planes of the observation. With the intents precomputed this
//                    pass is a few instructions per car and every lane of the warp has an env.
//
// Per-env shared state: tile descriptors, TEnv, intents (4 B / car), 16-bit car squares, optional 4-bit
// occupancy counters per square (envs with >= TK_OCC_MIN cars), the lane-column prefix of a new map, and
// the env's slice of the CTA's observation bitstring. Car lists live in HBM as [env][2][max_cars]: the
// tick reads the live half and writes the other one (order-stable compaction of despawned cars without
// hazards), then flips misc bit 15.
#pragma once
#include "pgtg_phases.cuh"

namespace pgtg {

#ifndef PGTG_TK_OCC_SAT
#define PGTG_TK_OCC_SAT 15  /* tests/emu also builds a variant that saturates at 3 to exercise the exact-count fallback */
#endif
constexpr int TK_OCC_SAT = PGTG_TK_OCC_SAT;  // a 4-bit per-square counter is exact below this value; at it, sticky "unknown"
constexpr int TK_OCC_MIN = 33;  // up to 32 cars the whole list is one warp step and needs no per-square counters

// intent word: kind 0-1 | target square x 2-9, y 10-17 | route 18-22 | delay 23-24 | push 25 | profile 26-28 | moved 31
enum : uint32_t { IK_STAY = 0, IK_LANE = 1, IK_ENTER = 2, IK_DESPAWN = 3, IK_PUSH = 1u << 25, IK_MOVED = 1u << 31 };
PG_HD uint32_t intent_pack(uint32_t kind, int tx, int ty, int route, int delay, bool push, int profile) {
  return kind | (uint32_t)tx << 2 | (uint32_t)ty << 10 | (uint32_t)route << 18 | (uint32_t)delay << 23 | (push ? IK_PUSH : 0u) | (uint32_t)profile << 26;
}
PG_HD unsigned intent_xy(uint32_t w) { return (w >> 2) & 0xFFFFu; }
PG_HD int intent_route(uint32_t w) { return (int)((w >> 18) & 31u); }
PG_HD int intent_delay(uint32_t w) { return (int)((w >> 23) & 3u); }
PG_HD int intent_profile(uint32_t w) { return (int)((w >> 26) & 7u); }

struct TEnv {
  EnvRegs e;
  uint64_t key;
  int32_t action, n_cars;        // cars when the tick starts (constant within an episode)
  int32_t tile_x, tile_y;        // the agent's tile before its move (rule engine, environment.py:208-224)
  int32_t in_tile;               // cars in that tile after the traffic advance
  uint32_t hist[5];              // their routes: 8-bit counter per route id
  int32_t hist_overflow;         // a route counter wrapped: the rule engine falls back to the list scan
  uint32_t ng_key;               // nearest remaining goal-line square of the position the next per-env phase asks about (d << 16 | x << 8 | y)
  uint64_t bloom;                // 64-bit filter over the squares that hold (or held, this tick) a car: a clear bit = no car there
  int32_t n_despawn;             // cars that leave the map in this tick (counted by the intent phase)
  int32_t done;                  // StepResult.outcome of this tick
  int32_t new_cars, num_positions, perm_h;  // initial traffic of the episode that starts in this tick
  uint32_t perm_keys[4];
};

struct TkShared {
  Lut* lut; uint2* spread;
  uint16_t* tiles;     // [G][tile_stride]
  TEnv* env;           // [G]
  uint32_t* intent;    // [G][MC]
  uint16_t* fxy;       // [G][MC] car squares: old ones until the resolve pass, final ones after it
  uint32_t* occ;       // [G][occ_words] 4-bit counters per square, 15 = sticky "unknown" (null when MC < TK_OCC_MIN)
  uint32_t* bits;      // CTA observation bitstring, env g at bit g * obs_bits
  uint16_t* colpre;    // [G][ncolp] lane squares of the tiles before t (new episodes)
  uint16_t* torg;      // [T] origin square of tile t (x | y << 8); [T] bytes after it: which map borders the tile touches (N 1, E 2, S 4, W 8)
  uint8_t* tborder;
  uint32_t* wbits;     // [32 warps][32] per-warp 1024-bit square filter of the resolve pass (zero between uses)
  uint8_t* item_g;     // [G * MC] item -> env of the CTA (the tick's cars, later the new episodes' cars)
  int* off;            // [G + 1] car items of the tick
  int* off2;           // [G + 1] car items of the episodes that start in this tick
  int* counters;       // [16]
  double* dsum;        // [2]
  int* done_list;      // [G]
  int bits_words, G, MC, occ_words, ncolp;
};
struct TkLayout {
  uint32_t lut, spread, tiles, env, intent, fxy, occ, bits, colpre, torg, tborder, wbits, item_g, off, off2, counters, dsum, done_list, total;
  int bits_words, G, MC, occ_words, ncolp;
};
PG_HOSTDEV TkLayout tk_layout(const DevCfg& c, int G) {
  TkLayout L;
  uint32_t o = 0;
  auto take = [&](size_t bytes) { uint32_t at = o; o += (uint32_t)align16(bytes); return at; };
  L.G = G; L.MC = c.max_cars;
  L.occ_words = c.max_cars >= TK_OCC_MIN ? (c.WS * c.HS + 7) / 8 : 0;
  L.ncolp = (c.T + 2) & ~1;
  L.bits_words = (G * c.obs_bits + 31) / 32 + 4;
  L.lut = take(sizeof(Lut)); L.spread = take(256 * sizeof(uint2));
  L.tiles = take(sizeof(uint16_t) * G * c.tile_stride);
  L.env = take(sizeof(TEnv) * G);
  L.intent = take(sizeof(uint32_t) * G * L.MC);
  L.fxy = take(sizeof(uint16_t) * G * L.MC);
  L.occ = take(sizeof(uint32_t) * G * L.occ_words);
  L.bits = take(sizeof(uint32_t) * L.bits_words);
  L.colpre = take(sizeof(uint16_t) * G * L.ncolp);
  L.torg = take(sizeof(uint16_t) * c.T); L.tborder = take((size_t)c.T);
  L.wbits = take(sizeof(uint32_t) * 32 * 32);
  L.item_g = take((size_t)G * L.MC);
  L.off = take(sizeof(int) * (G + 1)); L.off2 = take(sizeof(int) * (G + 1));
  L.counters = take(sizeof(int) * 16); L.dsum = take(sizeof(double) * 2);
  L.done_list = take(sizeof(int) * G);
  L.total = o;
  return L;
}
// whether the traffic tick can run a configuration with G envs per CTA; the others take the general (sequential) tick.
// (Large maps with dense traffic, or a wide sliding window with many planes, outgrow shared memory.)
PG_HOSTDEV bool tk_fits(const DevCfg& c, int G) { return tk_layout(c, G).total <= 220u * 1024u && c.max_cars <= 0xFFFF; }
PG_HOSTDEV TkShared tk_carve(unsigned char* base, const TkLayout& L) {
  TkShared s;
  s.lut = (Lut*)(base + L.lut); s.spread = (uint2*)(base + L.spread); s.tiles = (uint16_t*)(base + L.tiles);
  s.env = (TEnv*)(base + L.env); s.intent = (uint32_t*)(base + L.intent); s.fxy = (uint16_t*)(base + L.fxy);
  s.occ = L.occ_words ? (uint32_t*)(base + L.occ) : nullptr; s.bits = (uint32_t*)(base + L.bits);
  s.colpre = (uint16_t*)(base + L.colpre); s.torg = (uint16_t*)(base + L.torg); s.tborder = (uint8_t*)(base + L.tborder); s.wbits = (uint32_t*)(base + L.wbits); s.item_g = (uint8_t*)(base + L.item_g); s.off = (int*)(base + L.off); s.off2 = (int*)(base + L.off2);
  s.counters = (int*)(base + L.counters); s.dsum = (double*)(base + L.dsum); s.done_list = (int*)(base + L.done_list);
  s.bits_words = L.bits_words; s.G = L.G; s.MC = L.MC; s.occ_words = L.occ_words; s.ncolp = L.ncolp;
  return s;
}

PG_HD MapView tk_map(const DevCfg& c, const TkShared& sh, int g, bool with_goal_key = false) {
  MapView m = {c, *sh.lut, sh.tiles + g * c.tile_stride, sh.env[g].e.plan, nullptr, nullptr, nullptr, 0u, false};
  if (with_goal_key) { m.ng_key = sh.env[g].ng_key; m.ng_pre = true; }
  return m;
}
// nearest_goal (rule engine's heading, next_subgoal_direction) one TILE per thread: min over the tile's goal-line squares
// of the key, folded into the env's ng_key with a shared-memory atomicMin. The position asked about: the agent's.
PG_HD void tk_goal_key(const DevCfg& c, const TkShared& sh, int g, int tile, bool clamp) {
  TEnv& t = sh.env[g];
  const MapView m = tk_map(c, sh, g);
  int px = t.e.x, py = t.e.y;
  if (clamp) {  // get_observation clamps the position into the map first (:1352-1353)
    px = px < 0 ? 0 : (px > c.WS - 1 ? c.WS - 1 : px); py = py < 0 ? 0 : (py > c.HS - 1 ? c.HS - 1 : py);
  }
  const uint32_t k = m.tile_goal_key(tile, px, py);
  if (k != 0xFFFFFFFFu) pg_atomic_min(&t.ng_key, k);
}

// ---- 4-bit occupancy counters (exact below TK_OCC_SAT; at TK_OCC_SAT sticky = "count the list") ----------------
PG_HD int occ4_index(const DevCfg& c, unsigned xy) { return (int)(xy & 255u) * c.HS + (int)(xy >> 8); }
PG_HD int occ4_get(const uint32_t* o, int i) { return (int)((o[i >> 3] >> ((i & 7) * 4)) & 15u); }
PG_HD void occ4_inc(uint32_t* o, int i) {
  const int sh = (i & 7) * 4;
  if (((o[i >> 3] >> sh) & 15u) < (uint32_t)TK_OCC_SAT) o[i >> 3] += 1u << sh;
}
PG_HD void occ4_dec(uint32_t* o, int i) {
  const int sh = (i & 7) * 4;
  const uint32_t v = (o[i >> 3] >> sh) & 15u;
  if (v >= 1u && v < (uint32_t)TK_OCC_SAT) o[i >> 3] -= 1u << sh;
}
PG_HD void occ4_inc_atomic(uint32_t* o, int i) {
  const int sh = (i & 7) * 4;
  uint32_t* w = o + (i >> 3);
  uint32_t old = *(volatile uint32_t*)w;
  for (;;) {
    if (((old >> sh) & 15u) == (uint32_t)TK_OCC_SAT) return;
    const uint32_t seen = pg_atomic_cas(w, old, old + (1u << sh));
    if (seen == old) return;
    old = seen;
  }
}
PG_HD uint64_t bloom_bit(unsigned xy) { return 1ull << (((xy * 40503u) >> 10) & 63u); }
PG_HD bool tk_use_occ(const TkShared& sh, int n_cars) { return sh.occ_words != 0 && n_cars >= TK_OCC_MIN; }
PG_HD bool tk_scan(const uint16_t* fx, int n, unsigned xy) {
  for (int j = 0; j < n; j++)
    if (fx[j] == xy) return true;
  return false;
}

// per-CTA tile tables (stage, one tile per thread)
PG_HD void tk_stage_tile(const DevCfg& c, const TkShared& sh, int t) {
  const int tx = t % c.W, ty = t / c.W;
  sh.torg[t] = (uint16_t)(tx * TILE | (ty * TILE) << 8);
  sh.tborder[t] = (uint8_t)((ty == 0 ? 1u : 0u) | (tx == c.W - 1 ? 2u : 0u) | (ty == c.H - 1 ? 4u : 0u) | (tx == 0 ? 8u : 0u));
}
// build_spawner_list_tile_major (pgtg_logic.cuh) on the per-CTA tile tables: no divisions by the map width
PG_HD void tk_spawner_list(const DevCfg& c, const DevPtrs& p, const TkShared& sh, const MapView& m, int env) {
  int n = 0;
  uint16_t* list = p.spawners + (size_t)env * c.spawner_cap;
  for (int t = 0; t < c.T; t++) {
    const int ex = td_exits(m.tiles[t]);
    if (ex == 0) continue;  // no lanes on wall-only tiles (parser.py:113-118)
    unsigned slots = (m.L.native_spawner[ex] != 255 ? 1u : 0u) | (unsigned)(m.L.entry_ok[ex] & sh.tborder[t]) << 1;
    const unsigned org = sh.torg[t];
    while (slots) {
      const int k = pg_ffs(slots) - 1, sq = spawner_slot_square(m.L, ex, k);
      slots &= slots - 1;
      if (n < c.spawner_cap) list[n] = (uint16_t)(((org & 255u) + (unsigned)(sq / TILE)) | ((org >> 8) + (unsigned)(sq % TILE)) << 8);
      n++;
    }
  }
  p.spawner_count[env] = (uint16_t)(n < c.spawner_cap ? n : c.spawner_cap);
}

// ---- stage: one env per thread ----------------------------------------------------------------------
PG_HD void tk_stage_env(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env, int action) {
  TEnv& t = sh.env[g];
  EnvRegs e = load_regs(c, p, env);
  if (c.pregen) {  // the env's next map, should the episode end in this tick
    const size_t slot = (e.episode + 1u) & 1u;
    pg_prefetch_l2(p.next_tiles + (slot * c.N + (size_t)env) * c.T);
    pg_prefetch_l2(p.next_plan + slot * c.N + env);
  }
  if ((unsigned)action > 8u) { e.err |= 128; action = 4; }  // the reference would raise KeyError
  tick_prologue(c, e);
  t.e = e;
  t.key = p.key[env];
  t.action = action;
  t.n_cars = misc_ncars(e.misc);
  int tx = floordiv9(e.x), ty = floordiv9(e.y);
  t.tile_x = tx < 0 ? 0 : (tx > c.W - 1 ? c.W - 1 : tx);
  t.tile_y = ty < 0 ? 0 : (ty > c.H - 1 ? c.H - 1 : ty);
  t.in_tile = 0; t.n_despawn = 0; t.done = 0; t.new_cars = 0; t.num_positions = 0; t.perm_h = 2; t.hist_overflow = 0; t.bloom = 0; t.ng_key = 0xFFFFFFFFu;
#pragma unroll
  for (int i = 0; i < 5; i++) t.hist[i] = 0;
}
// exclusive prefix of a per-env count (thread g sums the envs before it; G <= 128) ...
// ... and the item -> env table of the flat phases that follow
PG_HD void tk_prefix(const TkShared& sh, int* off, int g, int nvalid, bool new_cars) {
  int s = 0;
  for (int j = 0; j < g; j++) s += new_cars ? sh.env[j].new_cars : sh.env[j].n_cars;
  off[g] = s;
  const int mine = new_cars ? sh.env[g].new_cars : sh.env[g].n_cars;
  for (int k = 0; k < mine; k++) sh.item_g[s + k] = (uint8_t)g;
  if (g == nvalid - 1) {
    s += mine;
    for (int j = nvalid; j <= sh.G; j++) off[j] = s;
  }
}

// ---- intents: one car per thread (_get_next_car_position_and_route, environment.py:881-968) -----------
PG_HD void tk_intent(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int r, int env) {
  TEnv& t = sh.env[g];
  const EnvRegs& e = t.e;
  const MapView m = tk_map(c, sh, g);
  const uint64_t rec = car_list(c, p, env, misc_half(e.misc))[r];
  const Car car = car_unpack(rec);
  const unsigned xy_old = car_xy(rec);
  sh.fxy[g * sh.MC + r] = (uint16_t)xy_old;
  if (tk_use_occ(sh, t.n_cars)) occ4_inc_atomic(sh.occ + g * sh.occ_words, occ4_index(c, xy_old));
  // _should_car_move (:678-691)
  uint32_t w0[4] = {0u, 0u, 0u, 0u}, w1[4];
  bool have1 = false, move = false;
  int delay = car.delay;
  if (delay > 0) delay--;
  else {
    philox_car_block(t.key, e.elapsed, e.episode, r, 0, w0);
    if (car_u32_to_uniform(w0[CW_DELAY]) < c.drv_reaction_delay[car.profile]) delay = 1 + (int)pg_umulhi(w0[CW_IDX], 3u);
    else move = car_u32_to_uniform(w0[CW_SPEED]) < c.drv_speed_multiplier[car.profile];
  }
  uint32_t word = intent_pack(IK_STAY, 0, 0, car.route, delay, false, car.profile);
  if (move) {
    bool found = false;
    const int ctx = car.x / TILE, cty = car.y / TILE, clx = car.x - ctx * TILE, cly = car.y - cty * TILE;
    // which neighbour square continues the journey (up, down, left, right, first match wins, :891-932): inside the car's
    // tile this is a table lookup per (tile type, square, route); only a move across a tile border looks at the other tile
    const unsigned m0 = pg_ldg(&p.step_lut[((size_t)td_exits(m.tiles[cty * c.W + ctx]) * 81 + clx * TILE + cly) * PGTG_NUM_ROUTE_IDS + car.route]);
    unsigned lane_mask = m0 & 15u, enter_mask = m0 >> 4;
    if (clx == 0 || cly == 0 || clx == TILE - 1 || cly == TILE - 1) {
#pragma unroll
      for (int d = 0; d < 4; d++) {
        const bool cross = d == 0 ? cly == 0 : d == 1 ? cly == TILE - 1 : d == 2 ? clx == 0 : clx == TILE - 1;
        if (!cross) continue;
        const int ntx = ctx + (d == 2 ? -1 : d == 3 ? 1 : 0), nty = cty + (d == 0 ? -1 : d == 1 ? 1 : 0);
        if (ntx < 0 || nty < 0 || ntx >= c.W || nty >= c.H) continue;  // inside_map
        const int nlx = d == 2 ? TILE - 1 : d == 3 ? 0 : clx, nly = d == 0 ? TILE - 1 : d == 1 ? 0 : cly;
        const unsigned tm = pg_ldg(&p.target_lut[((size_t)td_exits(m.tiles[nty * c.W + ntx]) * 81 + nlx * TILE + nly) * PGTG_NUM_ROUTE_IDS + car.route]);
        if ((tm >> (4 + d)) & 1u) enter_mask |= 1u << d;  // 'car_lane all d' wins over a lane of the same square (:915)
        else if ((tm >> d) & 1u) lane_mask |= 1u << d;
      }
    }
    if (lane_mask | enter_mask) {
      found = true;
      const int d = pg_ffs(lane_mask | enter_mask) - 1;
      int ntx = ctx, nty = cty, nlx = clx + (d == 2 ? -1 : d == 3 ? 1 : 0), nly = cly + (d == 0 ? -1 : d == 1 ? 1 : 0);
      if (nlx < 0) { nlx = TILE - 1; ntx--; } else if (nlx >= TILE) { nlx = 0; ntx++; }
      if (nly < 0) { nly = TILE - 1; nty--; } else if (nly >= TILE) { nly = 0; nty++; }
      const unsigned td = m.tiles[nty * c.W + ntx];
      const int ex = td_exits(td), sq = nlx * TILE + nly, px = ntx * TILE + nlx, py = nty * TILE + nly;
      if ((enter_mask >> d) & 1u) {  // entering a new tile: uniform new route, never blocked (:915-928)
        const uint64_t ld = lane_desc(ex, sq);
        const int n = ld_n(ld);
        word = intent_pack(IK_ENTER, px, py, ld_route(ld, n > 1 ? (int)pg_umulhi(w0[CW_IDX], (uint32_t)n) : 0), delay, false, car.profile);
      } else {
        bool stop = false;
        if (td_otype(td) == 4 && bit81(m.L.mask[td_omask(td)], sq) && !bit81(m.L.wall[ex], sq)) {  // a traffic light (:934-942)
          const int phase = light_phase(c, misc_light(e.misc));
          if (phase != 0) {
            philox_car_block(t.key, e.elapsed, e.episode, r, 1, w1);
            have1 = true;
            const double u = car_u32_to_uniform(w1[CW_LIGHT & 3]);
            stop = phase == 1 ? u < c.drv_yellow_stop[car.profile] : u >= c.drv_red_violation[car.profile];
          }
        }
        if (!stop) {
          const bool impatient = c.drv_min_following[car.profile] == 0 || (double)car.patience > c.drv_patience_threshold[car.profile];
          const bool push = impatient && car_u32_to_uniform(w0[CW_PUSH]) < c.drv_push_probability[car.profile];  // :950-958
          word = intent_pack(IK_LANE, px, py, car.route, delay, push, car.profile);
        }
      }
    }
    if (!found) {  // leaves the map; its replacement (_spawn_new_car, :970-1002) is appended to the list
      if (!have1) philox_car_block(t.key, e.elapsed, e.episode, r, 1, w1);
      int sx = 0, sy = 0;
      const int ns = p.spawner_count ? p.spawner_count[env] : 0;  // (no list on a handle created without traffic)
      if (ns > 0) {
        const unsigned v = p.spawners[(size_t)env * c.spawner_cap + (ns > 1 ? (int)pg_umulhi(w1[CW_SPAWNER & 3], (uint32_t)ns) : 0)];
        sx = (int)(v & 255u); sy = (int)(v >> 8);
      }
      const double u = car_u32_to_uniform(w1[CW_PROFILE & 3]);
      int prof = 0;
      while (prof < PGTG_NUM_PROFILES - 1 && c.profile_cdf[prof] <= u) prof++;
      const uint64_t sd = lane_desc(m.tile_type_at(sx, sy), m.local_sq(sx, sy));
      const int n = ld_n(sd);
      int route = 0;
      if (n == 0) pg_atomic_or(&t.e.err, 16u);
      else route = ld_route(sd, n > 1 ? (int)pg_umulhi(w1[CW_SPAWN_ROUTE & 3], (uint32_t)n) : 0);
      word = intent_pack(IK_DESPAWN, sx, sy, route, 0, false, prof);
      pg_atomic_add(&t.n_despawn, 1);
    }
  }
  sh.intent[g * sh.MC + r] = word;
}

// ---- resolve + commit: one env per WARP, 32 consecutive cars of its list per step --------------------------------
// Blocking in list order (environment.py:944-965, 1121-1127): car r is blocked iff some other car stands on its target
// square at ITS turn -- cars before it at their new squares (a replacement of a car that left the map included), cars
// after it at their old squares. Chunk by chunk (32 cars = 32 lanes):
//   count(r) = occ[T_r]                                   every car of the env at its current square (earlier chunks
//                                                         already final, this chunk and later ones still old)
//            + #{j < r in the chunk, moved: T_j == T_r}   arrived before r's turn
//            - #{j < r in the chunk, moved: old_j == T_r} left before r's turn
// Lanes whose target meets no old square of a lane of the chunk that may leave it (a 1024-bit per-warp filter) and no
// target of another lane (match_any) decide at once from occ; the few others are settled one by one in lane order
// with three ballots each. Envs with <= 32 cars need no occ array: the chunk is the whole list and occ[T_r] is a ballot.
// The chunk is then committed: live half -> other half of the car list, order-stable (a despawned car's replacement goes
// to the end of the list: slot n - n_despawn + rank), counters updated with shared-memory atomics.
PG_HD void occ4_dec_atomic(uint32_t* o, int i) {
  const int sh = (i & 7) * 4;
  uint32_t* w = o + (i >> 3);
  uint32_t old = *(volatile uint32_t*)w;
  for (;;) {
    const uint32_t v = (old >> sh) & 15u;
    if (v == 0u || v == (uint32_t)TK_OCC_SAT) return;
    const uint32_t seen = pg_atomic_cas(w, old, old - (1u << sh));
    if (seen == old) return;
    old = seen;
  }
}

PG_HD unsigned square_hash10(unsigned xy) { return ((xy * 40503u) >> 6) & 1023u; }

PG_HD void tk_resolve_commit(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env, int wslot) {
  PG_WARP_LANE
  TEnv& t = sh.env[g];
  const int n = t.n_cars, nd_total = t.n_despawn;
  uint32_t* it = sh.intent + g * sh.MC;
  uint16_t* fx = sh.fxy + g * sh.MC;
  const bool use_occ = tk_use_occ(sh, n);
  uint32_t* occ = use_occ ? sh.occ + g * sh.occ_words : nullptr;
  const int half = misc_half(t.e.misc);
  const uint64_t* A = car_list(c, p, env, half);
  uint64_t* B = car_list(c, p, env, half ^ 1);
  uint32_t* wb = sh.wbits + wslot * 32;
  uint32_t bloom_lo = 0, bloom_hi = 0;  // filter over the final squares (the agent's collision test)
  int nd_before = 0;
  for (int b = 0; b < n; b += 32) {
    PG_LV(uint32_t, w); PG_LV(unsigned, T); PG_LV(unsigned, old); PG_LV(int, moved); PG_LV(int, occv); PG_LV(uint32_t, same); PG_LV(uint32_t, hit);
    uint32_t inv;
    PG_FOR_LANES {
      const bool valid = b + l < n;
      LV(w) = valid ? it[b + l] : (uint32_t)IK_STAY;
      LV(T) = intent_xy(LV(w));
      LV(old) = valid ? (unsigned)fx[b + l] : 0x1FFFFu;
      const uint32_t kind = LV(w) & 3u;
      LV(occv) = (use_occ && kind == IK_LANE) ? occ4_get(occ, occ4_index(c, LV(T))) : 0;
      LV(moved) = kind == IK_ENTER || kind == IK_DESPAWN || (kind == IK_LANE && (LV(occv) == 0 || (LV(w) & IK_PUSH)));
    }
    // which lanes' turn order matters? Targets that meet the old square of a lane of this chunk that may leave it
    // (with counters: only movers matter, a staying occupant is in occ already; without: every old square, the filter
    // doubles as the occupancy test) or the target of another lane. 1024-bit filter per warp, exact on a miss.
    PG_FOR_LANES {
      const bool in = b + l < n && (!use_occ || LV(moved) || (LV(w) & 3u) == IK_LANE);
      if (in) { const unsigned h = square_hash10(LV(old)); pg_atomic_or(&wb[h >> 5], 1u << (h & 31u)); }
    }
    PG_SYNCWARP();
    PG_MATCH_ANY(same, (LV(w) & 3u) != IK_STAY ? LV(T) : 0x20000u + (uint32_t)l);
    PG_FOR_LANES {
      const unsigned h = square_hash10(LV(T));
      LV(hit) = (wb[h >> 5] >> (h & 31u)) & 1u;
    }
    PG_BALLOT(inv, (LV(w) & 3u) == IK_LANE && ((LV(hit) && (!use_occ || LV(occv) > 0)) || LV(occv) == TK_OCC_SAT || (LV(same) & (LV(same) - 1u)) != 0));
    PG_SYNCWARP();
    PG_FOR_LANES { wb[l] = 0; }
    while (inv) {  // the lanes whose turn order matters, in list order
      const int rl = pg_ffs(inv) - 1;
      inv &= inv - 1;
      const unsigned Tr = intent_xy(it[b + rl]);
      uint32_t occm, arrm, leftm;
      PG_BALLOT(occm, LV(old) == Tr);
      PG_BALLOT(arrm, l < rl && LV(moved) && LV(T) == Tr);
      PG_BALLOT(leftm, l < rl && LV(moved) && LV(old) == Tr);
      int base = (int)pg_popc(occm);
      if (use_occ) {
        base = occ4_get(occ, occ4_index(c, Tr));
        if (base == TK_OCC_SAT) {  // counter saturated: count the list itself (chunks before this one final, the rest old)
          base = 0;
          for (int jb = 0; jb < n; jb += 32) { uint32_t m; PG_BALLOT(m, jb + l < n && (unsigned)fx[jb + l] == Tr); base += (int)pg_popc(m); }
        }
      }
      const bool blocked = base + (int)pg_popc(arrm) - (int)pg_popc(leftm) > 0;
      PG_FOR_LANES { if (l == rl) LV(moved) = !blocked || (LV(w) & IK_PUSH) != 0; }
    }
    uint32_t desm, fin_lo, fin_hi;
    PG_BALLOT(desm, (LV(w) & 3u) == IK_DESPAWN);
    PG_FOR_LANES {
      const int r = b + l;
      if (r < n) {
        const uint32_t kind = LV(w) & 3u;
        const unsigned fin = LV(moved) ? LV(T) : LV(old);
        if (LV(moved)) {
          fx[r] = (uint16_t)fin;
          if (use_occ) { occ4_dec_atomic(occ, occ4_index(c, LV(old))); occ4_inc_atomic(occ, occ4_index(c, fin)); }
        }
        Car car = car_unpack(A[r]);
        const int before = nd_before + (int)pg_popc(desm & ((1u << l) - 1u));  // cars ahead of r that left the map
        int slot;
        if (kind == IK_DESPAWN) {  // its replacement (_spawn_new_car, :970-1002) goes to the end of the list
          slot = n - nd_total + before;
          car.id = t.e.next_car_id + (unsigned)before;
          car.route = intent_route(LV(w)); car.profile = intent_profile(LV(w)); car.patience = 0; car.delay = 0;
        } else {
          slot = r - before;
          car.delay = intent_delay(LV(w));
          if (LV(moved)) { car.patience = 0; car.route = intent_route(LV(w)); }
          else car.patience++;
        }
        car.x = (int)(fin & 255u); car.y = (int)(fin >> 8);
        B[slot] = car_pack(car);
        if (c.num_rules > 0 && car.x / TILE == t.tile_x && car.y / TILE == t.tile_y) {  // the rule engine's view of the agent's tile
          pg_atomic_add(&t.in_tile, 1);
          const uint32_t prev = pg_atomic_add(&t.hist[car.route >> 2], 1u << (8 * (car.route & 3)));
          if (((prev >> (8 * (car.route & 3))) & 255u) == 255u) t.hist_overflow = 1;  // > 255 cars of one route in one tile
        }
      }
    }
    PG_REDUCE_OR(fin_lo, b + l < n ? (uint32_t)bloom_bit(LV(moved) ? LV(T) : LV(old)) : 0u);
    PG_REDUCE_OR(fin_hi, b + l < n ? (uint32_t)(bloom_bit(LV(moved) ? LV(T) : LV(old)) >> 32) : 0u);
    bloom_lo |= fin_lo; bloom_hi |= fin_hi;
    nd_before += (int)pg_popc(desm);
    PG_SYNCWARP();  // the next chunk reads the counters this one updated
  }
  PG_FOR_LANES { if (l == 0) t.bloom = (uint64_t)bloom_hi << 32 | bloom_lo; }
}

// ---- the agent's part of the tick: one env per thread -----------------------------------------------------
struct ExtTraffic {
  static constexpr bool external = true;
  const TkShared* sh;
  int g;
  PG_MEMBER bool braking(const DevCfg& c, const DevPtrs& p, const MapView& m, const EnvRegs& e, int env, int n_cars) const {
    // apply_braking / evaluate_rule (environment.py:226-294) on the counters the commit phase collected
    if (c.num_rules == 0 || !(n_cars > 0 || c.rules_without_traffic)) return false;
    const TEnv& t = sh->env[g];
    if (t.hist_overflow) return apply_braking(c, p, m, e, env);  // 8-bit route counters wrapped: fall back to the list scan
    const int type = td_exits(m.tiles[t.tile_y * c.W + t.tile_x]);
    const double speed = sqrt((double)(e.vx * e.vx + e.vy * e.vy));
    int adir = -1;
    for (int i = 0; i < c.num_rules; i++) {
      const pgtg_rule& rule = p.rules[i];
      if (type != rule.tile_type) continue;
      if (!(rule.vel_lo <= speed && speed <= rule.vel_hi)) continue;
      if (t.in_tile < rule.min_traffic) continue;
      if (adir < 0) adir = agent_direction(c, p, m, e);
      int matching = 0;
      for (int q = 0; q < PGTG_NUM_ROUTE_IDS; q++) matching += (int)((t.hist[q >> 2] >> (8 * (q & 3))) & 255u) * rule.weight[adir][q];
      if (matching >= rule.min_matching_traffic) return true;
    }
    return false;
  }
  PG_MEMBER bool car_at(const DevCfg& c, const DevPtrs&, const EnvRegs&, int, int x, int y, int n_cars) const {
    const unsigned xy = (unsigned)x | (unsigned)y << 8;
    if (!(sh->env[g].bloom & bloom_bit(xy))) return false;
    const uint16_t* fx = sh->fxy + g * sh->MC;
    if (tk_use_occ(*sh, n_cars)) {
      const int v = occ4_get(sh->occ + g * sh->occ_words, occ4_index(c, xy));
      return v == TK_OCC_SAT ? tk_scan(fx, n_cars, xy) : v != 0;
    }
    return tk_scan(fx, n_cars, xy);
  }
};

PG_HD StepResult tk_agent(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env) {
  TEnv& t = sh.env[g];
  EnvRegs& e = t.e;
  e.next_car_id += (uint32_t)t.n_despawn;
  e.misc ^= 1u << 15;  // the commit phase wrote the other half: it is the live list now
  MapView m = tk_map(c, sh, g, true);  // (ng_key: nearest goal-line square of the position before the move)
  ExtTraffic tr = {&sh, g};
  StepResult r = env_step<PGTG_RNG_PHILOX, false, ExtTraffic>(c, p, m, e, env, t.action, tr);
  write_step_outputs<false>(c, p, env, e, r);
  t.done = r.outcome;
  return r;
}

// ---- observation ---------------------------------------------------------------------------------------
// the traffic plane bit of one car (environment.py:1397-1409) in the observation of an agent at (ex, ey)
PG_HD void tk_car_bit(const DevCfg& c, uint32_t* bits, uint32_t base, int ex, int ey, unsigned xy) {
  const int ch = c.kind_channel[PGTG_CH_TRAFFIC];
  if (ch < 0) return;
  const int cx = (int)(xy & 255u), cy = (int)(xy >> 8);
  if (!c.sliding) {
    const int pix = ex < 0 ? 0 : (ex > c.WS - 1 ? c.WS - 1 : ex), piy = ey < 0 ? 0 : (ey > c.HS - 1 ? c.HS - 1 : ey);
    const int lx = cx - (pix / TILE) * TILE, ly = cy - (piy / TILE) * TILE;
    if (lx >= 0 && lx < TILE && ly >= 0 && ly < TILE) emit_bits(bits, base + (uint32_t)(ch * 81 + lx * TILE + ly), 1u);
  } else {
    const int ix = cx - (ex - c.window_k), iy = cy - (ey - c.window_k);
    if (ix >= 0 && ix < c.P && iy >= 0 && iy < c.P) emit_bits(bits, base + (uint32_t)(ch * c.P * c.P + ix * c.P + iy), 1u);
  }
}
// sliding window: one (plane, window column) per thread
PG_HD void tk_sliding_column(const DevCfg& c, const TkShared& sh, int g, int item) {
  const int ch = item / c.P, ix = item - ch * c.P, kind = c.channel_kind[ch];
  if (kind == PGTG_CH_ZERO || kind == PGTG_CH_TRAFFIC) return;  // (the traffic plane comes from the car threads)
  const EnvRegs& e = sh.env[g].e;
  const MapView m = tk_map(c, sh, g);
  const uint32_t col = sliding_column_bits(c, m, kind, light_phase(c, misc_light(e.misc)), e.x - c.window_k + ix, e.y - c.window_k);
  emit_bits(sh.bits, (uint32_t)g * (uint32_t)c.obs_bits + (uint32_t)(ch * c.P * c.P + ix * c.P), col);
}
// map planes + scalars of env g (the traffic plane comes from the car threads); final = terminal observation
PG_HD void tk_emit(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env, bool final_obs) {
  const TEnv& t = sh.env[g];
  EnvRegs e = t.e;
  e.misc &= 0xFFFFu;  // no cars for env_observe's own traffic loop
  const MapView m = tk_map(c, sh, g, c.use_nsd != 0);  // (ng_key: ... of the position observed)
  int32_t pos[2], vel[2], nsd;
  env_observe<false>(c, p, m, e, env, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, pos, vel, &nsd, !c.sliding);  // (sliding planes: tk_sliding_column)
  if (final_obs) {
    p.f_obs_position[2 * env] = pos[0]; p.f_obs_position[2 * env + 1] = pos[1];
    p.f_obs_velocity[2 * env] = vel[0]; p.f_obs_velocity[2 * env + 1] = vel[1];
    if (c.use_nsd) p.f_obs_nsd[env] = nsd;
    return;
  }
  write_obs_scalars_and_state<false>(c, p, sh.tiles + g * c.tile_stride, env, t.e, pos, vel, nsd);
}

// ---- reset of a finished env: one env per thread (PGTGEnv.reset, environment.py:581-656, minus the cars) ------
// part A: the map and the agent
template <int TMAX, bool PREGEN>
PG_HD void tk_reset_map(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env) {
  TEnv& t = sh.env[g];
  EnvRegs& e = t.e;
  MapView m = tk_map(c, sh, g);
  if (PREGEN) env_reset_pregenerated<PGTG_RNG_PHILOX, false, true>(c, p, m, e, env);
  else env_reset<PGTG_RNG_PHILOX, TMAX, true>(c, p, m, e, env);
}
// part B, three independent pieces that different warps run side by side on the new map:
// 1 the lane squares (how many cars, _create_initial_traffic :833-834), 2 the car_spawners list, 4 the placement keys
PG_HD void tk_reset_traffic(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int env, int parts) {
  TEnv& t = sh.env[g];
  EnvRegs& e = t.e;
  const MapView m = tk_map(c, sh, g);
  if (!(c.traffic_density > 0)) {  // a car-free configuration on this tick (sliding window / next_subgoal_direction): nothing to prepare
    if (parts & 1) { t.num_positions = 0; t.new_cars = 0; e.misc = misc_pack(0, 0, 0, 0); e.next_car_id = 0; }
    return;
  }
  if (parts & 2) tk_spawner_list(c, p, sh, m, env);
  if (parts & 4) philox_car_block(t.key, e.elapsed, e.episode, -1, 0, t.perm_keys);
  if (parts & 1) {
    const int np = lane_tile_prefix(c, m, sh.colpre + g * sh.ncolp);
    int nc = initial_car_count(c, np);
    if (nc > c.max_cars) { e.err |= 32; nc = c.max_cars; }
    t.num_positions = np; t.new_cars = nc; t.perm_h = feistel_bits(np);
    e.misc = misc_pack(0, 0, nc, 0);
    e.next_car_id = (uint32_t)nc;  // ids follow the slots (_create_initial_traffic, :830-879)
  }
}
// one car of the new episode per thread
PG_HD void tk_new_car(const DevCfg& c, const DevPtrs& p, const TkShared& sh, int g, int j, int env) {
  TEnv& t = sh.env[g];
  const MapView m = tk_map(c, sh, g);
  const int idx = initial_car_position(t.perm_keys, t.perm_h, t.num_positions, j);
  int x, y;
  lane_square_tile_major(c, m, sh.colpre + g * sh.ncolp, idx, x, y);
  uint32_t w[4];
  philox_car_block(t.key, t.e.elapsed, t.e.episode, j, 0, w);
  const double u = car_u32_to_uniform(w[CW0_PROFILE]);
  Car car;
  car.profile = 0;
  while (car.profile < PGTG_NUM_PROFILES - 1 && c.profile_cdf[car.profile] <= u) car.profile++;
  const uint64_t d = lane_desc(m.tile_type_at(x, y), m.local_sq(x, y));
  const int n = ld_n(d);
  car.route = 0;
  if (n == 0) pg_atomic_or(&p.error[env], 16u);  // (straight to HBM: the env's own thread may be past its emit)
  else car.route = ld_route(d, n > 1 ? (int)pg_umulhi(w[CW0_ROUTE], (uint32_t)n) : 0);
  car.id = (unsigned)j; car.x = x; car.y = y; car.patience = 0; car.delay = 0;
  car_list(c, p, env, 0)[j] = car_pack(car);
  tk_car_bit(c, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, t.e.x, t.e.y, (unsigned)x | (unsigned)y << 8);
}

}  // namespace pgtg
