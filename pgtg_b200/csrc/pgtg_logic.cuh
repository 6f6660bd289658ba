// pgtg_logic.cuh -- the per-env game logic: one tick, one reset (incl. procedural map generation),
// and the observation planes, all on the packed tile-descriptor representation.
// Compiled by nvcc into the kernels of pgtg_kernels.cu (and by g++ into tests/emu, see
// pgtg_device.cuh). Reference citations are paths under /root/reference/pgtg/.
#pragma once
#include "pgtg_device.cuh"

namespace pgtg {

PG_HD int select32(uint32_t v, int n);

// car lists: [env][half][slot]; `half` = misc bit 15 (the live list), the other half is scratch / write target
PG_HD uint64_t* car_list(const DevCfg& c, const DevPtrs& p, int env, int half) { return p.cars + ((size_t)env * 2 + half) * c.max_cars; }

PG_HD int light_phase(const DevCfg& c, int counter) {  // environment.py:1004-1015: 0 green 1 yellow 2 red
  return counter < c.light_green ? 0 : (counter < c.light_green + c.light_yellow ? 1 : 2);
}

// ---------------------------------------------------------------------------------------------
// car spawners: squares carrying "car_spawner", enumerated in the x-major order of
// EpisodeMap.__init__ (map.py:31-42) without materialising the list.
// sets bit sq of an 81-bit bitmap held in three registers (no dynamic indexing: that would push the
// array into local memory)
PG_HD void or_bit81(uint32_t w[3], int sq) {
  uint32_t b = 1u << (sq & 31);
  int i = sq >> 5;
  w[0] |= i == 0 ? b : 0u; w[1] |= i == 1 ? b : 0u; w[2] |= i == 2 ? b : 0u;
}

PG_HD void spawner_bits(const DevCfg& c, const Lut& L, int ex, int tx, int ty, uint32_t out[3]) {
  out[0] = out[1] = out[2] = 0;
  if (ex == 0) return;  // no lanes on wall-only tiles (parser.py:113-118)
  int ns = L.native_spawner[ex];
  if (ns != 255) or_bit81(out, ns);
  // border tiles: tile-entry squares 'car_lane all <inward>' (parser.py:120-148)
  if (tx == 0) { int sq = L.entry_sq[3]; if (ld_all(lane_desc(ex, sq)) == 4) or_bit81(out, sq); }
  if (tx == c.W - 1) { int sq = L.entry_sq[2]; if (ld_all(lane_desc(ex, sq)) == 3) or_bit81(out, sq); }
  if (ty == 0) { int sq = L.entry_sq[1]; if (ld_all(lane_desc(ex, sq)) == 2) or_bit81(out, sq); }
  if (ty == c.H - 1) { int sq = L.entry_sq[0]; if (ld_all(lane_desc(ex, sq)) == 1) or_bit81(out, sq); }
}
PG_HD uint32_t col9(const uint32_t w[3], int lx) {  // the 9 bits of local column lx
  int b = lx * TILE, wi = b >> 5, sh = b & 31;  // selects, not w[wi]: keeps the bitmap in registers
  uint32_t lo = wi == 0 ? w[0] : wi == 1 ? w[1] : w[2], hi = wi == 0 ? w[1] : wi == 1 ? w[2] : 0u;
  uint32_t v = lo >> sh;
  if (sh > 23) v |= hi << (32 - sh);
  return v & 0x1FFu;
}
// Build the env's car_spawner list (x-major order of EpisodeMap.__init__, map.py:31-42) once per
// episode: _spawn_new_car (environment.py:977-979) then indexes it in O(1).
PG_HDN void build_spawner_list(const DevCfg& c, const DevPtrs& p, const MapView m, int env) {
  int n = 0;
  for (int tx = 0; tx < c.W; tx++)
    for (int lx = 0; lx < TILE; lx++) {
      if (!((m.L.spawner_cols >> lx) & 1)) continue;
      for (int ty = 0; ty < c.H; ty++) {
        uint32_t sb[3];
        spawner_bits(c, m.L, td_exits(m.tiles[ty * c.W + tx]), tx, ty, sb);
        uint32_t col = col9(sb, lx);
        while (col) {
          int ly = pg_ffs(col) - 1;
          col &= col - 1;
          if (n < c.spawner_cap) p.spawners[(size_t)env * c.spawner_cap + n] = (uint16_t)((tx * TILE + lx) | (ty * TILE + ly) << 8);
          n++;
        }
      }
    }
  p.spawner_count[env] = (uint16_t)(n < c.spawner_cap ? n : c.spawner_cap);
}

// Philox specification of the two index spaces the car stream draws from (the reference's x-major lists are only
// reproduced in the tape / numpy modes): both enumerate TILE BY TILE (t = ty * W + tx ascending), which needs no
// scan over the 9W x 9H squares:
//   lane squares   within a tile by local square index lx * 9 + ly ascending;
//   car spawners   within a tile by slot: 0 the tile type's native spawner (dead ends), then the border spawners of
//                  the north, east, south and west map border (slots 1-4; parser.py:120-148).
PG_HD unsigned spawner_slots(const DevCfg& c, const Lut& L, int ex, int tx, int ty) {  // 5-bit slot mask of tile (tx, ty)
  if (ex == 0) return 0u;  // no lanes on wall-only tiles (parser.py:113-118)
  unsigned border = (ty == 0 ? 1u : 0u) | (tx == c.W - 1 ? 2u : 0u) | (ty == c.H - 1 ? 4u : 0u) | (tx == 0 ? 8u : 0u);
  return (L.native_spawner[ex] != 255 ? 1u : 0u) | (L.entry_ok[ex] & border) << 1;
}
PG_HD int spawner_slot_square(const Lut& L, int ex, int slot) {  // local square of a slot
  return slot == 0 ? L.native_spawner[ex] : L.entry_sq[slot == 1 ? 1 : slot == 2 ? 2 : slot == 3 ? 0 : 3];
}
PG_HD void build_spawner_list_tile_major(const DevCfg& c, const DevPtrs& p, const MapView& m, int env) {
  int n = 0;
  uint16_t* list = p.spawners + (size_t)env * c.spawner_cap;
  for (int t = 0; t < c.T; t++) {
    const int ex = td_exits(m.tiles[t]), tx = t % c.W, ty = t / c.W;
    unsigned slots = spawner_slots(c, m.L, ex, tx, ty);
    while (slots) {
      const int k = pg_ffs(slots) - 1, sq = spawner_slot_square(m.L, ex, k);
      slots &= slots - 1;
      if (n < c.spawner_cap) list[n] = (uint16_t)((tx * TILE + sq / TILE) | (ty * TILE + sq % TILE) << 8);
      n++;
    }
  }
  p.spawner_count[env] = (uint16_t)(n < c.spawner_cap ? n : c.spawner_cap);
}
// lane squares tile by tile: tpre[t] = lane squares of the tiles before t (T + 1 entries); returns the total
PG_HD int lane_tile_prefix(const DevCfg& c, const MapView& m, uint16_t* tpre) {
  int n = 0;
  for (int t = 0; t < c.T; t++) { tpre[t] = (uint16_t)n; n += m.L.lane_count[td_exits(m.tiles[t])]; }
  tpre[c.T] = (uint16_t)n;
  return n;
}
PG_HD void lane_square_tile_major(const DevCfg& c, const MapView& m, const uint16_t* tpre, int idx, int& x, int& y) {
  int lo = 0, hi = c.T;  // last tile with tpre[t] <= idx
  while (hi - lo > 1) { int mid = (lo + hi) >> 1; if ((int)tpre[mid] <= idx) lo = mid; else hi = mid; }
  const uint32_t* la = m.L.lane_any[td_exits(m.tiles[lo])];
  int rest = idx - tpre[lo], sq = 0;
#pragma unroll
  for (int w = 0; w < 3; w++) {
    uint32_t bits = la[w];
    const int cnt = pg_popc(bits);
    if (rest >= 0 && rest < cnt) { sq = w * 32 + select32(bits, rest); rest = -1; }
    else if (rest >= 0) rest -= cnt;
  }
  x = (lo % c.W) * TILE + sq / TILE; y = (lo / c.W) * TILE + sq % TILE;
}

// occupancy grid: per-tick 2-bit counters of the cars on every square (exact while < 3; the value 3
// is sticky and means "unknown, scan the list"). "Is there a car on (x, y)?" becomes O(1) instead
// of a scan over the car list -- the list scans were 70 % of the tick at ~230 cars per env.
constexpr int OCC_MIN_CARS = 32;
PG_HD int occ_get(const DevCfg& c, const DevPtrs& p, int env, int x, int y) {
  int i = x * c.HS + y;
  return (int)((p.occ[(size_t)(i >> 4) * c.N + env] >> ((i & 15) * 2)) & 3u);
}
PG_HD void occ_add(const DevCfg& c, const DevPtrs& p, int env, int x, int y) {
  int i = x * c.HS + y, sh = (i & 15) * 2;
  uint32_t& w = p.occ[(size_t)(i >> 4) * c.N + env];
  if (((w >> sh) & 3u) < 3u) w += 1u << sh;
}
PG_HD void occ_sub(const DevCfg& c, const DevPtrs& p, int env, int x, int y) {
  int i = x * c.HS + y, sh = (i & 15) * 2;
  uint32_t& w = p.occ[(size_t)(i >> 4) * c.N + env];
  uint32_t v = (w >> sh) & 3u;
  if (v == 1u || v == 2u) w -= 1u << sh;  // 3 stays 3
}

// ---------------------------------------------------------------------------------------------
// traffic (environment.py:658-691, 830-1002, 1121-1127)
template <int RNG>
PG_HD int random_route_at(const MapView& m, Rng<RNG>& rng, EnvRegs& e, int x, int y, int slot, int pos) {
  uint64_t d = lane_desc(m.tile_type_at(x, y), m.local_sq(x, y));
  int n = ld_n(d);
  if (n == 0) { e.err |= 16; return 0; }
  return ld_route(d, rng.car_index(slot, pos, n));  // sorted route names, car_rng.choice (:861-874)
}

PG_HD bool any_car_at(const uint64_t* list, unsigned xy, int lo, int hi) {
  for (int k = lo; k < hi; k++)
    if (car_xy(list[k]) == xy) return true;
  return false;
}

// one car tick; returns false when the car leaves the map (None at environment.py:968)
template <int RNG>
PG_HD bool car_next(const DevCfg& c, const DevPtrs& p, const MapView& m, EnvRegs& e, Rng<RNG>& rng, int env, Car& car,
                     int r, int w, int n, int s, bool use_occ, const uint64_t* live, const uint64_t* scratch) {
  // _should_car_move (:678-691)
  bool move;
  if (car.delay > 0) { car.delay--; move = false; }
  else if (rng.car_uniform(r, CW_DELAY) < c.drv_reaction_delay[car.profile]) { car.delay = 1 + rng.car_index(r, CW_IDX, 3); move = false; }
  else move = rng.car_uniform(r, CW_SPEED) < c.drv_speed_multiplier[car.profile];
  if (!move) { car.patience++; return true; }
#pragma unroll 1
  for (int d = 0; d < 4; d++) {  // up, down, left, right (:891-902)
    int px = car.x + (d == 2 ? -1 : d == 3 ? 1 : 0), py = car.y + (d == 0 ? -1 : d == 1 ? 1 : 0);
    if (!m.inside(px, py)) continue;
    uint64_t ld = lane_desc(m.tile_type_at(px, py), m.local_sq(px, py));
    if (ld == 0) continue;
    if (ld_all(ld) == d + 1) {  // entering a new tile: uniform new route (:915-928)
      car.patience = 0;
      car.route = ld_route(ld, rng.car_index(r, CW_IDX, ld_n(ld)));
      car.x = px; car.y = py;
      return true;
    }
    int nl = ld_n(ld);
    for (int i = 0; i < nl; i++) {
      if (ld_route(ld, i) != car.route || ld_dir(ld, i) != d) continue;  // :932
      if (m.light_at(px, py)) {  // :934-942
        int phase = light_phase(c, misc_light(e.misc));
        bool stop = false;
        if (phase == 1) stop = rng.car_uniform(r, CW_LIGHT) < c.drv_yellow_stop[car.profile];
        else if (phase == 2) stop = rng.car_uniform(r, CW_LIGHT) >= c.drv_red_violation[car.profile];
        if (stop) { car.patience++; return true; }
      }
      // cars_on_next_position over the live list: survivors [0,w), not-yet-moved (r,n), and the
      // replacements spawned earlier this tick (scratch half) (:944-948)
      unsigned xy = (unsigned)px | (unsigned)py << 8;
      int occ = use_occ ? occ_get(c, p, env, px, py) : 3;
      bool blocked = occ == 1 || occ == 2;
      if (occ == 3)
        blocked = any_car_at(live, xy, 0, w) || any_car_at(live, xy, r + 1, n) || any_car_at(scratch, xy, 0, s);
      if (blocked) {  // :950-962
        if (c.drv_min_following[car.profile] == 0 || (double)car.patience > c.drv_patience_threshold[car.profile]) {
          if (rng.car_uniform(r, CW_PUSH) < c.drv_push_probability[car.profile]) { car.patience = 0; car.x = px; car.y = py; return true; }
        }
        car.patience++;
        return true;
      }
      car.patience = 0; car.x = px; car.y = py;  // :964-965
      return true;
    }
  }
  car.patience++;
  return false;
}

// The traffic tick is a cold, self-contained unit: it is the only consumer of the car stream
// during a tick, so it owns its Rng; the env registers travel by value so that the (hot,
// traffic-free) caller keeps everything in registers.
struct TrafficIO {
  uint32_t next_car_id, err;
  int64_t cursor;
};
template <int RNG>
PG_HDN TrafficIO advance_cars(const DevCfg& c, const DevPtrs& p, const MapView m, const EnvRegs e_in, int env) {
  // environment.py:1121-1127. Order-stable in place: survivors are compacted to [0,w), replacements
  // are parked in the scratch half in spawn order and appended afterwards (w + s == n).
  EnvRegs e = e_in;
  Rng<RNG> rng(p, e, env);
  int n = misc_ncars(e.misc), w = 0, s = 0;
  uint64_t* live = car_list(c, p, env, misc_half(e.misc));
  uint64_t* scratch = car_list(c, p, env, misc_half(e.misc) ^ 1);
  const bool use_occ = n >= OCC_MIN_CARS;
  if (use_occ) {  // rebuild the occupancy counters for this tick
    for (int i = 0; i < c.occ_words; i++) p.occ[(size_t)i * c.N + env] = 0;
    for (int r = 0; r < n; r++) { unsigned xy = car_xy(live[r]); occ_add(c, p, env, (int)(xy & 255), (int)(xy >> 8)); }
  }
  for (int r = 0; r < n; r++) {
    Car car = car_unpack(live[r]);
    int ox = car.x, oy = car.y;
    if (car_next<RNG>(c, p, m, e, rng, env, car, r, w, n, s, use_occ, live, scratch)) {
      if (use_occ && (car.x != ox || car.y != oy)) { occ_sub(c, p, env, ox, oy); occ_add(c, p, env, car.x, car.y); }
      live[w++] = car_pack(car);
    } else {  // _spawn_new_car (:970-1002)
      if (use_occ) occ_sub(c, p, env, ox, oy);
      int sx = 0, sy = 0;
      int ns = p.spawner_count ? p.spawner_count[env] : 0;  // (no list on a handle created without traffic: cars injected by set_state)
      if (!p.spawner_count) e.err |= 16;
      if (ns > 0) {
        unsigned v = p.spawners[(size_t)env * c.spawner_cap + rng.car_index(r, CW_SPAWNER, ns)];
        sx = (int)(v & 255); sy = (int)(v >> 8);
      }
      if (use_occ) occ_add(c, p, env, sx, sy);
      Car nc;
      nc.profile = rng.car_choice_cdf(r, CW_PROFILE, c.profile_cdf, PGTG_NUM_PROFILES);
      nc.route = random_route_at<RNG>(m, rng, e, sx, sy, r, CW_SPAWN_ROUTE);
      nc.id = e.next_car_id++;
      nc.x = sx; nc.y = sy; nc.patience = 0; nc.delay = 0;
      scratch[s++] = car_pack(nc);
    }
  }
  for (int i = 0; i < s; i++) live[w + i] = scratch[i];
  rng.flush();
  TrafficIO io;
  io.next_car_id = e.next_car_id; io.err = e.err; io.cursor = e.cursor;
  return io;
}

// lane squares per global column, x-major (traffic_spawnable_positions, map.py:35-38): colpre[X] = number of
// lane squares in the columns before X; returns their total. colpre has 9 W + 1 entries.
PG_HD int lane_column_prefix(const DevCfg& c, const MapView& m, uint16_t* colpre) {
  int ncol = c.W * TILE, num_positions = 0;
  for (int X = 0; X < ncol; X++) {
    colpre[X] = (uint16_t)num_positions;
    int tx = X / TILE, lx = X - tx * TILE;
    for (int ty = 0; ty < c.H; ty++) num_positions += pg_popc(col9(m.L.lane_any[td_exits(m.tiles[ty * c.W + tx])], lx));
  }
  colpre[ncol] = (uint16_t)num_positions;
  return num_positions;
}
// the idx-th lane square of that list
PG_HD void lane_square_at(const DevCfg& c, const MapView& m, const uint16_t* colpre, int idx, int& x, int& y) {
  int lo = 0, hi = c.W * TILE;  // last column with colpre[X] <= idx
  while (hi - lo > 1) { int mid = (lo + hi) >> 1; if ((int)colpre[mid] <= idx) lo = mid; else hi = mid; }
  int X = lo, tx = X / TILE, lx = X - tx * TILE, rest = idx - colpre[X];
  x = X; y = 0;
  for (int ty = 0; ty < c.H; ty++) {
    uint32_t col = col9(m.L.lane_any[td_exits(m.tiles[ty * c.W + tx])], lx);
    int cnt = pg_popc(col);
    if (rest < cnt) { while (rest--) col &= col - 1; y = ty * TILE + pg_ffs(col) - 1; break; }
    rest -= cnt;
  }
}
PG_HD int initial_car_count(const DevCfg& c, int num_positions) {  // int(len(spawnable) * density) (:833-834)
  int num_cars = (int)((double)num_positions * c.traffic_density);
  return num_cars > num_positions ? num_positions : num_cars;
}

template <int RNG>
PG_HDN uint32_t create_initial_traffic(const DevCfg& c, const DevPtrs& p, const MapView m, const EnvRegs e_in, int env, uint32_t car_words,
                                      int64_t* cursor_out, uint32_t* err_out) {
  // _create_initial_traffic (environment.py:830-879). Cold, self-contained unit (registers by value).
  EnvRegs e = e_in;
  Rng<RNG> rng(p, e, env);
  (void)car_words;
  uint16_t colpre[PGTG_MAX_TILES + 1];  // (>= 9 * 16 + 1) column prefix of the x-major list, or tile prefix in Philox mode
  int num_positions = RNG == PGTG_RNG_PHILOX ? lane_tile_prefix(c, m, colpre) : lane_column_prefix(c, m, colpre);
  int num_cars = initial_car_count(c, num_positions);
  if (num_cars > c.max_cars) { e.err |= 32; num_cars = c.max_cars; }
  uint64_t* live = car_list(c, p, env, misc_half(e.misc));
  if (num_cars > 0) {
    // car_rng.choice(n, size=k, replace=False): k distinct indices, kept raw in the car slots first
    if (RNG == PGTG_RNG_NUMPY) {
      // Generator.choice(n, size=k, replace=False): Floyd's sampling (membership via a bitmap in the occupancy
      // words, numpy uses a hash set) followed by the in-place shuffle of the k values
      for (int i = 0; i < (num_positions + 31) / 32; i++) p.occ[(size_t)i * c.N + env] = 0;
      for (int t = 0; t < num_cars; t++) {
        uint32_t j = (uint32_t)(num_positions - num_cars + t);
        uint32_t v = rng.np_bounded(PGTG_STREAM_CAR, j);
        uint32_t& wv = p.occ[(size_t)(v >> 5) * c.N + env];
        if ((wv >> (v & 31)) & 1u) { v = j; p.occ[(size_t)(j >> 5) * c.N + env] |= 1u << (j & 31); }
        else wv |= 1u << (v & 31);
        live[t] = (uint64_t)v;
      }
      for (int i = num_cars - 1; i >= 1; i--) {
        int jj = (int)rng.np_bounded(PGTG_STREAM_CAR, (uint32_t)i);
        uint64_t a = live[i];
        live[i] = live[jj];
        live[jj] = a;
      }
    } else if (RNG == PGTG_RNG_TAPE) {
      for (int j = 0; j < num_cars; j++) {
        int v = (int)rng.tape_next(PGTG_STREAM_CAR, PGTG_DRAW_INDEX);
        if (v < 0 || v >= num_positions) { e.err |= 4; v = 0; }
        live[j] = (uint64_t)(uint32_t)v;
      }
    } else {  // Philox specification: keyed Feistel permutation of the lane squares (pgtg_device.cuh, CW_*)
      uint32_t keys[4];
      philox_car_block(p.key[env], e.elapsed, e.episode, -1, 0, keys);
      const int m_bits = feistel_bits(num_positions);
      for (int j = 0; j < num_cars; j++) live[j] = (uint64_t)(uint32_t)initial_car_position(keys, m_bits, num_positions, j);
    }
    for (int j = 0; j < num_cars; j++) {
      int x, y;
      if (RNG == PGTG_RNG_PHILOX) lane_square_tile_major(c, m, colpre, (int)live[j], x, y);
      else lane_square_at(c, m, colpre, (int)live[j], x, y);
      Car car;
      car.profile = rng.car_choice_cdf(j, CW0_PROFILE, c.profile_cdf, PGTG_NUM_PROFILES);
      car.route = random_route_at<RNG>(m, rng, e, x, y, j, CW0_ROUTE);
      car.id = e.next_car_id++;
      car.x = x; car.y = y; car.patience = 0; car.delay = 0;
      live[j] = car_pack(car);
    }
  }
  rng.flush();
  *cursor_out = e.cursor; *err_out = e.err;
  return (uint32_t)num_cars | e.next_car_id << 16;
}

// ---------------------------------------------------------------------------------------------
// rule engine (environment.py:162-294)
PG_HD int floordiv9(int a) { return a >= 0 ? a / TILE : -((-a + TILE - 1) / TILE); }

PG_HDN int agent_direction(const DevCfg& c, const DevPtrs& p, const MapView m, const EnvRegs e) {
  // get_agent_direction (:185-206) over _get_subgoal_compass_directions (:1037-1090)
  int gx, gy;
  if (m.nearest_goal(e.x, e.y, gx, gy)) {
    int dx = gx - e.x, dy = gy - e.y;
    if (!(abs(dx) <= c.window_k && abs(dy) <= c.window_k)) {
      int R = c.lut_radius;
      int o = pg_ldg(&p.dirlut[(dy + R) * (2 * R + 1) + (dx + R)]) & 7;  // host-evaluated atan2 sector
      return o >> 1;  // N,NE -> s2n; E,SE -> w2e; S,SW -> n2s; W,NW -> e2w
    }
  }
  return (e.vx == 0 && e.vy == 0) ? PGTG_AGENT_STATIONARY : PGTG_AGENT_NEAR_GOAL;  // norm < 0.1
}

PG_HDN bool apply_braking(const DevCfg& c, const DevPtrs& p, const MapView m, const EnvRegs e, int env) {
  // apply_braking / evaluate_rule (:226-294)
  int n = misc_ncars(e.misc);
  if (c.num_rules == 0) return false;
  int tx = floordiv9(e.x), ty = floordiv9(e.y);
  tx = tx < 0 ? 0 : (tx > c.W - 1 ? c.W - 1 : tx);
  ty = ty < 0 ? 0 : (ty > c.H - 1 ? c.H - 1 : ty);
  int type = td_exits(m.tiles[ty * c.W + tx]);
  double speed = sqrt((double)(e.vx * e.vx + e.vy * e.vy));
  int adir = -1;
  for (int i = 0; i < c.num_rules; i++) {
    const pgtg_rule& rule = p.rules[i];
    if (type != rule.tile_type) continue;
    if (!(rule.vel_lo <= speed && speed <= rule.vel_hi)) continue;
    int in_tile = 0;
    const uint64_t* live = car_list(c, p, env, misc_half(e.misc));
    for (int k = 0; k < n; k++) {
      unsigned xy = car_xy(live[k]);
      if ((int)(xy & 255) / TILE == tx && (int)(xy >> 8) / TILE == ty) in_tile++;
    }
    if (in_tile < rule.min_traffic) continue;
    if (adir < 0) adir = agent_direction(c, p, m, e);
    int matching = 0;
    for (int k = 0; k < n; k++) {
      uint64_t cv = live[k];
      unsigned xy = car_xy(cv);
      if ((int)(xy & 255) / TILE == tx && (int)(xy >> 8) / TILE == ty) matching += rule.weight[adir][(cv >> 16) & 31];
    }
    if (matching >= rule.min_matching_traffic) return true;
  }
  return false;
}

// ---------------------------------------------------------------------------------------------
// one tick (environment.py:1092-1281)
struct StepResult {
  double reward, cost;
  int terminated, braking, outcome;  // outcome: 0 running, 1 crash, 2 final goal (3 truncated, set by phase_step)
  double ep_return;                  // return of the episode that just finished (phase_step)
  double ep_disc;                    // ... and its discounted return (evaluator statistics, when enabled)
};

PG_HD bool visited_test_set(const DevCfg& c, const DevPtrs& p, int env, int x, int y, bool set) {
  int idx = (x + 1) * c.vis_w + (y + 1);
  uint32_t& w = p.visited[(size_t)(idx >> 5) * c.N + env];
  bool was = (w >> (idx & 31)) & 1u;
  if (set) w |= 1u << (idx & 31);
  return was;
}

// How the agent's part of the tick sees the traffic. SeqTraffic = the sequential tick: the cars advance inside
// env_step, "is a car there" scans the list / the global occupancy counters. The warp-parallel traffic tick
// (pgtg_traffic.cuh) advances the cars beforehand and answers from shared memory (external = true).
struct SeqTraffic {
  static constexpr bool external = false;
  PG_MEMBER bool braking(const DevCfg& c, const DevPtrs& p, const MapView& m, const EnvRegs& e, int env, int n_cars) const {
    return (n_cars > 0 || c.rules_without_traffic) && apply_braking(c, p, m, e, env);  // the default rules need traffic in the agent's tile
  }
  PG_MEMBER bool car_at(const DevCfg& c, const DevPtrs& p, const EnvRegs& e, int env, int x, int y, int n_cars) const {
    int occ = n_cars >= OCC_MIN_CARS ? occ_get(c, p, env, x, y) : 3;
    if (occ == 3) return any_car_at(car_list(c, p, env, misc_half(e.misc)), (unsigned)x | (unsigned)y << 8, 0, n_cars);
    return occ != 0;
  }
};

// the first lines of PGTGEnv.step: tick counter and traffic-light counter (:1113-1115)
PG_HD void tick_prologue(const DevCfg& c, EnvRegs& e) {
  e.elapsed++;
  int light = misc_light(e.misc) + 1;  // the counter is below the period except after an arbitrary set_state
  if (light >= c.light_total) light = light == c.light_total ? 0 : light % c.light_total;
  e.misc = misc_pack(misc_flat(e.misc), light, misc_ncars(e.misc), misc_half(e.misc));
}

// LEAN = compile-time promise of the plain configuration (no traffic and no rule that can fire
// without it, fixed window written kind by kind, no next_subgoal_direction / visited penalty /
// cost split): the corresponding code is not even emitted, which is what keeps the hot kernel small.
template <int RNG, bool LEAN = false, class TR = SeqTraffic>
PG_HD StepResult env_step(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, int env, int action, const TR tr = TR()) {
  const bool split_cost = LEAN ? false : (bool)c.separate_reward_cost;
  StepResult r;
  r.reward = 0; r.cost = 0; r.terminated = 0; r.braking = 0; r.outcome = 0;
  double perf = 0;
  if (!TR::external) tick_prologue(c, e);
  const int light = misc_light(e.misc);
  int ax = action / 3 - 1, ay = action % 3 - 1;  // constants.py:6-16
  const int n_cars = LEAN ? 0 : misc_ncars(e.misc);
  if (!TR::external && n_cars > 0) {  // :1121-1127
    TrafficIO io = advance_cars<RNG>(c, p, m, e, env);
    e.next_car_id = io.next_car_id; e.err |= io.err; e.cursor = io.cursor;
  }
  Rng<RNG> rng(p, e, env);  // ice / broken road / sand streams of this tick
  int cx = e.x, cy = e.y;
  e.vx += ax; e.vy += ay;  // :1139
  if (!LEAN && tr.braking(c, p, m, e, env, n_cars)) { r.braking = 1; e.vx = 0; e.vy = 0; }  // :1145

  // _decompose_velocity (:693-748), produced lazily one unit sub-step at a time; the float64
  // rounding of _round(i * m) is reproduced with explicitly unfused IEEE operations
  int dx = e.vx, dy = e.vy;
  int adx = abs(dx), ady = abs(dy);
  int n_sub = adx > ady ? adx : ady;
  int sgx = (dx > 0) - (dx < 0), sgy = (dy > 0) - (dy < 0);
  double slope = 0.0;
  if (dx != 0 && dy != 0) slope = adx >= ady ? pg_ddiv((double)dy, (double)adx) : pg_ddiv((double)dx, (double)ady);
  int pxp = 0, pyp = 0;
  bool red = light_phase(c, light) == 2;
  int flat = misc_flat(e.misc);
  for (int i = 1; i <= n_sub + 1; i++) {
    int sx = 0, sy = 0;
    bool has_part = i <= n_sub;
    if (has_part) {
      int px, py;
      if (dx == 0) { px = 0; py = i * sgy; }
      else if (dy == 0) { px = i * sgx; py = 0; }
      else if (adx >= ady) { px = i * sgx; py = (int)floor(pg_dadd(pg_dmul((double)i, slope), 0.5)); }
      else { py = i * sgy; px = (int)floor(pg_dadd(pg_dmul((double)i, slope), 0.5)); }
      sx = px - pxp; sy = py - pyp; pxp = px; pyp = py;
    }
    // crash: off-map, wall, or a car on the square (:1158-1171)
    bool inside = m.inside(cx, cy);
    unsigned f = inside ? m.features(cx, cy) : (unsigned)SF_WALL;
    bool crash = !inside || (f & SF_WALL);
    if (!crash && !c.ignore_traffic_collisions && n_cars > 0) crash = tr.car_at(c, p, e, env, cx, cy, n_cars);
    if (crash) {
      if (split_cost) r.cost += c.crash_penalty; else r.reward -= c.crash_penalty;
      r.terminated = 1; r.outcome = 1;
      break;
    }
    if (f & SF_FINAL) {  // :1174-1180
      double isr = c.sum_subgoals_reward / (double)plan_ns(e.plan);  // :631-633
      if (split_cost) perf += isr + c.final_goal_bonus; else r.reward += isr + c.final_goal_bonus;
      r.terminated = 1; r.outcome = 2;
      break;
    }
    if (f & SF_SUBGOAL) {  // :1183-1188
      double isr = c.sum_subgoals_reward / (double)plan_ns(e.plan);
      if (split_cost) perf += isr; else r.reward += isr;
      m.consume_subgoal(cx, cy);
      e.flags |= EF_TILES_DIRTY;
    }
    if (!has_part) continue;  // :1191-1192
    int nx = cx + sx, ny = cy + sy;  // red light on the NEXT square, before ice (:1195-1202)
    if (red && m.inside(nx, ny) && m.light_at(nx, ny)) {
      if (split_cost) r.cost += c.light_penalty; else r.reward -= c.light_penalty;
    }
    if ((f & SF_ICE) && rng.uniform(PGTG_STREAM_ICE) < c.ice_p) {  // :1205-1213
      int ia = rng.index(PGTG_STREAM_ICE, 9);
      sx = ia / 3 - 1; sy = ia % 3 - 1;
    }
    if ((f & SF_BROKEN) && rng.uniform(PGTG_STREAM_BROKEN) < c.broken_p) flat = 1;  // :1216-1223
    if ((f & SF_SAND) && rng.uniform(PGTG_STREAM_SAND) < c.sand_p) {  // :1226-1234
      cx += sx; cy += sy; e.vx = 0; e.vy = 0;
      break;
    }
    cx += sx; cy += sy;  // :1236
  }
  if (flat) { e.vx = 0; e.vy = 0; }  // :1240-1241
  e.misc = misc_pack(flat, light, misc_ncars(e.misc), misc_half(e.misc));
  if (!LEAN && c.vis_words) {  // :1244-1255
    bool was = visited_test_set(c, p, env, cx, cy, true);
    if (was && !(ax == 0 && ay == 0)) {
      if (split_cost) r.cost += c.visited_penalty; else r.reward -= c.visited_penalty;
    }
  }
  if (c.standing_penalty != 0 && ax == 0 && ay == 0 && e.x == cx && e.y == cy) {  // :1257-1263
    if (split_cost) r.cost += c.standing_penalty; else r.reward -= c.standing_penalty;
  }
  e.x = cx; e.y = cy;
  rng.flush();
  if (split_cost) r.reward = perf;  // :1271-1281
  return r;
}

// ---------------------------------------------------------------------------------------------
// procedural map generation (map_generator.py:43-472) on bitboards. TMAX (16 / 64 / 256) is the
// compile-time bound on the tile count: it sizes the boards (one 32-bit word for the default 4x4
// map), the alive mask of removable edges and the BFS scratch, so the default case runs entirely
// in registers.
template <int TMAX>
struct Board {
  static constexpr int NW = (TMAX + 31) / 32;
  uint32_t w[NW];
};
template <int TMAX> PG_HD bool bget(const Board<TMAX>& b, int i) {
  if (Board<TMAX>::NW == 1) return (b.w[0] >> i) & 1u;
  return (b.w[i >> 5] >> (i & 31)) & 1u;
}
template <int TMAX> PG_HD void bset(Board<TMAX>& b, int i) {
  if (Board<TMAX>::NW == 1) b.w[0] |= 1u << i; else b.w[i >> 5] |= 1u << (i & 31);
}
template <int TMAX> PG_HD void bclr(Board<TMAX>& b, int i) {
  if (Board<TMAX>::NW == 1) b.w[0] &= ~(1u << i); else b.w[i >> 5] &= ~(1u << (i & 31));
}
template <int TMAX> PG_HD void bzero(Board<TMAX>& b) {
#pragma unroll
  for (int k = 0; k < Board<TMAX>::NW; k++) b.w[k] = 0;
}

// position of the n-th (0-based) set bit, n < popc(v): popcount binary search, no loop
PG_HD int select32(uint32_t v, int n) {
  int pos = 0, cnt;
  cnt = pg_popc(v & 0xFFFFu); if (n >= cnt) { n -= cnt; pos += 16; v >>= 16; }
  cnt = pg_popc(v & 0xFFu); if (n >= cnt) { n -= cnt; pos += 8; v >>= 8; }
  cnt = pg_popc(v & 0xFu); if (n >= cnt) { n -= cnt; pos += 4; v >>= 4; }
  cnt = pg_popc(v & 0x3u); if (n >= cnt) { n -= cnt; pos += 2; v >>= 2; }
  if (n >= (int)(v & 1u)) pos += 1;
  return pos;
}

// Does removing edge (a, b) keep start and goal connected? E bit i: edge i<->i+1, S bit i: edge
// i<->i+W (the edge is already cleared). Flood from a: reaching b means nothing changed (early
// exit, typically after going round one grid face); otherwise the flood ends on a's whole
// component and the graph stays start-goal connected iff s and g are on the same side.
// start-goal connectivity of a <= 32-tile subgraph by flood fill (builds the connectivity table)
PG_HD bool flood_connected32(int W, uint32_t e, uint32_t so, int s, int g) {
  if (s == g) return true;
  uint32_t reach = 1u << s, goal = 1u << g;
  for (;;) {
    uint32_t nx = reach | ((reach & e) << 1) | ((reach >> 1) & e) | ((reach & so) << W) | ((reach >> W) & so);
    if (nx & goal) return true;
    if (nx == reach) return false;
    reach = nx;
  }
}

template <int TMAX>
PG_HD bool still_connected(const DevCfg& c, const DevPtrs& p, const Board<TMAX>& E, const Board<TMAX>& S, int a, int b, int s, int g) {
  if (TMAX <= 32) {  // whole board in one register: flood fill by shifts
    uint32_t e = E.w[0], so = S.w[0], reach = 1u << a, tb = 1u << b;
    for (;;) {
      uint32_t nx = reach | ((reach & e) << 1) | ((reach >> 1) & e) | ((reach & so) << c.W) | ((reach >> c.W) & so);
      if (nx & tb) return true;
      if (nx == reach) return ((reach >> s) & 1u) == ((reach >> g) & 1u);
      reach = nx;
    }
  } else if (TMAX <= 64) {
    uint64_t e = (uint64_t)E.w[0] | (uint64_t)E.w[1] << 32, so = (uint64_t)S.w[0] | (uint64_t)S.w[1] << 32;
    uint64_t reach = 1ull << a, tb = 1ull << b;
    for (;;) {
      uint64_t nx = reach | ((reach & e) << 1) | ((reach >> 1) & e) | ((reach & so) << c.W) | ((reach >> c.W) & so);
      if (nx & tb) return true;
      if (nx == reach) return ((reach >> s) & 1ull) == ((reach >> g) & 1ull);
      reach = nx;
    }
  } else {
    Board<TMAX> seen;
    bzero(seen);
    uint8_t q[TMAX];
    int qh = 0, qt = 0;
    bset(seen, a); q[qt++] = (uint8_t)a;
    while (qh < qt) {
      int n = q[qh++];
      if (n == b) return true;
      int cand[4] = {n - c.W, n + 1, n + c.W, n - 1};
      bool ok[4] = {n >= c.W && bget(S, n - c.W), bget(E, n), bget(S, n), n > 0 && bget(E, n - 1)};
      for (int k = 0; k < 4; k++)
        if (ok[k] && !bget(seen, cand[k])) { bset(seen, cand[k]); q[qt++] = (uint8_t)cand[k]; }
    }
    return bget(seen, s) == bget(seen, g);
  }
}

template <int RNG>
PG_HD void random_border_position(const DevCfg& c, Rng<RNG>& rng, int& x, int& y) {
  // chose_random_start_or_goal_position (map_generator.py:600-626)
  switch (rng.index(PGTG_STREAM_MAP, 4)) {
    case 0: x = rng.index(PGTG_STREAM_MAP, c.W); y = 0; break;
    case 1: x = c.W - 1; y = rng.index(PGTG_STREAM_MAP, c.H); break;
    case 2: x = rng.index(PGTG_STREAM_MAP, c.W); y = c.H - 1; break;
    default: x = 0; y = rng.index(PGTG_STREAM_MAP, c.H); break;
  }
}
template <int RNG>
PG_HD int random_direction(const DevCfg& c, Rng<RNG>& rng, int x, int y) {
  // chose_random_start_or_goal_direction (:571-597): candidates in north, east, south, west order
  int d[4], n = 0;
  if (y == 0) d[n++] = 0;
  if (x == c.W - 1) d[n++] = 1;
  if (y == c.H - 1) d[n++] = 2;
  if (x == 0) d[n++] = 3;
  int k = rng.index(PGTG_STREAM_MAP, n);
  return k == 0 ? d[0] : k == 1 ? d[1] : k == 2 ? d[2] : d[3];
}

template <int RNG>
PG_HD void choose_start_goal(const DevCfg& c, Rng<RNG>& rng, int& sx, int& sy, int& sd, int& gx, int& gy, int& gd) {
  // chose_random_start_and_goal_position_and_direction (:475-568)
  if (c.start_mode == 2) random_border_position<RNG>(c, rng, sx, sy);
  if (c.goal_mode == 2) random_border_position<RNG>(c, rng, gx, gy);
  if (c.min_sg_dist >= 0)
    while (abs(sx - gx) + abs(sy - gy) < c.min_sg_dist) {
      random_border_position<RNG>(c, rng, sx, sy);
      random_border_position<RNG>(c, rng, gx, gy);
    }
  if (c.start_mode != 0) sd = random_direction<RNG>(c, rng, sx, sy);
  if (c.goal_mode != 0) gd = random_direction<RNG>(c, rng, gx, gy);
  while (sx == gx && sy == gy && sd == gd) {
    if (c.start_mode == 2) random_border_position<RNG>(c, rng, sx, sy);
    if (c.start_mode != 0) sd = random_direction<RNG>(c, rng, sx, sy);
    if (c.goal_mode == 2) random_border_position<RNG>(c, rng, gx, gy);
    if (c.goal_mode != 0) gd = random_direction<RNG>(c, rng, gx, gy);
  }
}

// connectivity-table index -> E / S boards (E has a hole after every row, S is contiguous)
PG_HD void graph_to_boards(const DevCfg& c, uint32_t graph, uint32_t& E, uint32_t& S) {
  uint32_t e = 0, rowmask = (1u << (c.W - 1)) - 1u;
  for (int r = 0; r < c.H; r++) e |= ((graph >> (r * (c.W - 1))) & rowmask) << (r * c.W);
  E = e; S = graph >> c.conn_ne;
}

// Philox specification of the edge removal (generate_map_graph, map_generator.py:245-264). Each trip picks uniformly among
// the grid edges not tried yet -- exactly what the reference's draw over removable_edges amounts to (both directions of an
// edge are listed and leave the list together, :249-253). The edges are numbered in the order of the connectivity-table
// bits (horizontal edges row by row, then vertical edges by tile) and kept in an array, a[i] = i at the start; a trip
// takes ONE word of the map stream (also when a single edge is left), i = (word * n) >> 32 over the n edges still in the
// array, tries edge a[i] and closes the gap with the last one (a[i] = a[n-1], n -= 1): a Fisher-Yates walk, every trip
// productive, no k-th-set-bit select and no rejected draws (map generation is bound by its chain of dependent lookups).
PG_HOSTDEV int edge_chunk_bits(int n_edges) { int b = 1; while (b < 31 && (1 << b) < n_edges) b++; return b; }

// the loop for grids of <= 32 edges with the connectivity table: the edge set is the table index itself. `arr`: n_edges
// bytes (rounded up to a word) of this thread's scratch. The stream must stand at a block boundary (it does: TABLED maps have a fixed start and
// goal, nothing was drawn before); four trips per Philox block, unrolled.
template <int RNG>
PG_HD uint32_t remove_edges_tabled(const DevCfg& c, const DevPtrs& p, Rng<RNG>& rng, uint8_t* arr) {
  const int n_und = c.H * (c.W - 1) + c.W * (c.H - 1);
  uint32_t graph = (c.conn_bits >= 32 ? 0u : (1u << c.conn_bits)) - 1u;
  for (int i = 0; 4 * i < n_und; i++) ((uint32_t*)arr)[i] = 0x03020100u + 0x04040404u * (uint32_t)i;  // a[i] = i (arr is word-aligned, room for 4 * ceil(n / 4))
  int n = n_und;
  int go = n > 0 ? 2 * n_und - c.edges_to_keep : 0;  // :245 (both directions of an edge are counted): > 0 = carry on
  uint32_t pos = rng.position(PGTG_STREAM_MAP);
  while (go > 0) {
    uint32_t w[4];
    rng.block(PGTG_STREAM_MAP, pos >> 2, w);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (go > 0) {
        const int i = (int)pg_umulhi(w[k], (uint32_t)n);  // :249
        const int edge = arr[i];
        const uint32_t pbit = 1u << edge;
        arr[i] = arr[n - 1];
        n--; pos++;
        // "start and goal still connected?" is a pure function of the edge set: one lookup in the 2^E-bit table built
        // once per handle (2 MB for the 4x4 grid, L2-resident) -- unless one of the two grid faces next to the edge is
        // otherwise intact: then its end points stay connected round that face and nothing can change (half of the
        // trips; the generation is bound by the L2's rate of scattered sector requests, so this halves its time)
        const uint32_t g2 = graph & ~pbit;
        const uint2 face = pg_ldg(&p.face_tab[edge]);
        bool keep = (graph & face.x) == face.x || (graph & face.y) == face.y;
        if (!keep) keep = (pg_ldg(&p.conn_table[g2 >> 5]) >> (g2 & 31)) & 1u;
        graph = keep ? g2 : graph;
        go = n > 0 ? 2 * pg_popc(graph) - c.edges_to_keep : 0;
      }
    }
  }
  rng.set_position(PGTG_STREAM_MAP, pos);
  return graph;
}

// Philox specification of add_connections_to_borders (map_generator.py:337-371): `border_connections` distinct slots out of
// n (host-table order, default start / goal slots removed), which is a uniformly random subset -- drawn by rejection:
// the stream's next words are cut into chunks of ceil(log2 n) bits, lowest first, floor(32 / bits) per word, the rest of
// a word dropped; a chunk >= n or naming a chosen slot is skipped. Returns
// the chosen slots as a bit set (the order of the picks does not matter: each sets one exit bit).
template <int RNG, typename MASK = uint64_t>
PG_HD MASK choose_border_slots(const DevCfg& c, Rng<RNG>& rng) {
  const int n = c.n_border_slots;
  int left = c.border_connections < n ? c.border_connections : n;
  MASK chosen = 0;
  if (left <= 0) return chosen;
  const int cbits = edge_chunk_bits(n), per_word = 32 / cbits;
  const uint32_t cmask = (1u << cbits) - 1u;
  const MASK valid = n >= (int)(8 * sizeof(MASK)) ? ~(MASK)0 : (((MASK)1 << n) - 1);
  while (left > 0) {
    uint32_t cw = rng.word(PGTG_STREAM_MAP);
    for (int k = 0; k < per_word && left > 0; k++) {
      const MASK bit = (MASK)1 << (cw & cmask);  // :367 (callers with a 32-bit mask have <= 32 slots, so cbits <= 5)
      cw >>= cbits;
      if (bit & valid & ~chosen) { chosen |= bit; left--; }
    }
  }
  return chosen;
}

// add_obstacles_to_map (map_generator.py:374-472) for one tile with exits `ex`: one random() whatever the outcome (:415),
// then the obstacle type (:418) and its mask (:430, :470). Returns the descriptor bits type << 4 | mask << 7 (0 = none).
template <int RNG>
PG_HD unsigned obstacle_draw(const DevCfg& c, Rng<RNG>& rng, int ex) {
  const double u = rng.uniform(PGTG_STREAM_MAP);  // :415
  if (!(u < c.obstacle_probability) || ex == 0) return 0u;
  const int type = 1 + rng.choice_cdf(PGTG_STREAM_MAP, c.obstacle_cdf, 4);  // :418
  int mask;
  if (type != 4) mask = rng.index(PGTG_STREAM_MAP, 8);  // :430
  else {
    // candidate masks 8..13 as a bit set (no indexed local array: that would live in local memory)
    const int cnt = pg_popc(ex);
    unsigned cand = (unsigned)(ex & 15);                          // 8..11: one light per exit
    if ((ex & 1) && (ex & 4) && cnt >= 3) cand |= 16u;            // 12: north-south pair
    if ((ex & 2) && (ex & 8) && cnt >= 3) cand |= 32u;            // 13: east-west pair
    int k = rng.index(PGTG_STREAM_MAP, pg_popc(cand));  // :470
    while (k-- > 0) cand &= cand - 1;                             // drop the k lowest candidates
    mask = 8 + pg_ffs(cand) - 1;
  }
  return (unsigned)(type << 4 | mask << 7);
}

// TABLED = compile-time promise that both per-handle tables exist (fixed start/goal, <= 16 tiles,
// <= 24 inner edges): the flood fill, the BFS and the start/goal draws are not emitted.
template <int RNG, int TMAX, bool TABLED = false>
PG_HD void generate_map(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, Rng<RNG>& rng) {
  int sx = c.start_x, sy = c.start_y, sd = c.start_dir, gx = c.goal_x, gy = c.goal_y, gd = c.goal_dir;
  if (!TABLED && (c.start_mode != 0 || c.goal_mode != 0)) choose_start_goal<RNG>(c, rng, sx, sy, sd, gx, gy, gd);
  int W = c.W, T = c.T;
  int st = sy * W + sx, gt = gy * W + gx;

  // generate_map_graph (:192-266). The full grid (host-built masks); an edge picked from
  // removable_edges (edges() order, host table) stays removed iff start and goal remain connected
  // -- which is what the reference's "on the BFS path? then is_connected? else restore" amounts
  // to, independent of BFS tie-breaking (SURVEY.md a13).
  Board<TMAX> E, S;
#pragma unroll
  for (int k = 0; k < Board<TMAX>::NW; k++) { E.w[k] = c.full_e[k]; S.w[k] = c.full_s[k]; }
  // with the connectivity table the graph is kept as the table index itself (one bit per grid edge)
  const bool tabled = TABLED || (TMAX <= 32 && c.conn_bits != 0);
  uint32_t graph = tabled ? ((c.conn_bits >= 32 ? 0u : (1u << c.conn_bits)) - 1u) : 0u;
  if (RNG == PGTG_RNG_PHILOX) {
    // Philox specification: see remove_edges_tabled above (one word per trip, Fisher-Yates walk over the edge array)
    constexpr int UW = (2 * TMAX + 31) / 32;
    if (UW == 1 && tabled && (rng.position(PGTG_STREAM_MAP) & 3u) == 0u) {
      alignas(4) uint8_t arr8[32];
      graph = remove_edges_tabled<RNG>(c, p, rng, arr8);
    } else {
    uint16_t arr[2 * TMAX];  // (the slow path: big maps, random start / goal -- a local-memory array is fine here)
    const int n_he = c.H * (W - 1), n_und = n_he + W * (c.H - 1);
    for (int i = 0; i < n_und; i++) arr[i] = (uint16_t)i;
    int n = n_und, cur = 2 * n_und;
    while (cur > c.edges_to_keep && n > 0) {  // :245
      const int i = (int)pg_umulhi(rng.word(PGTG_STREAM_MAP), (uint32_t)n);  // :249
      const int pos = arr[i];
      arr[i] = arr[n - 1];
      n--;
      if (tabled) {
        const uint32_t g2 = graph & ~(1u << pos);
        const bool keep = (pg_ldg(&p.conn_table[g2 >> 5]) >> (g2 & 31)) & 1u;
        graph = keep ? g2 : graph;
        cur -= keep ? 2 : 0;
        continue;
      }
      const bool horiz = pos < n_he;
      const int lo = horiz ? (pos / (W - 1)) * W + pos % (W - 1) : pos - n_he;
      const int a = lo, b = horiz ? lo + 1 : lo + W;
      if (horiz) bclr(E, lo); else bclr(S, lo);
      if (still_connected<TMAX>(c, p, E, S, a, b, st, gt)) cur -= 2;
      else { if (horiz) bset(E, lo); else bset(S, lo); }
    }
    }
  } else {
  constexpr int AW = (4 * TMAX + 31) / 32;
  uint32_t alive[AW];
  int n_tab = c.n_edge_tab, n_alive = n_tab, cur = n_tab;
#pragma unroll
  for (int i = 0; i < AW; i++) alive[i] = (i * 32 + 32 <= n_tab) ? 0xFFFFFFFFu : (i * 32 < n_tab ? ((1u << (n_tab & 31)) - 1u) : 0u);
  while (cur > c.edges_to_keep && n_alive > 0) {  // :245
    int idx = rng.index(PGTG_STREAM_MAP, n_alive);  // :249
    int i;
    if (AW == 2) {  // default 4x4 map: 48 directed edges in two registers
      int pc0 = pg_popc(alive[0]);
      bool hi = idx >= pc0;
      i = select32(hi ? alive[1] : alive[0], hi ? idx - pc0 : idx) + (hi ? 32 : 0);
    } else {
      int wi = 0;
      for (;; wi++) { int pc = pg_popc(alive[wi]); if (idx < pc) break; idx -= pc; }
      i = wi * 32 + select32(alive[wi], idx);
    }
    unsigned rv = m.edge_rev[i];
    int j = rv & 1023;
    if (AW == 2) {
      uint64_t clr = ~((1ull << i) | (1ull << j));
      alive[0] &= (uint32_t)clr; alive[1] &= (uint32_t)(clr >> 32);
    } else {
      alive[i >> 5] &= ~(1u << (i & 31));
      alive[j >> 5] &= ~(1u << (j & 31));
    }
    n_alive -= 2;
    if (tabled) {
      // "start and goal still connected?" is a pure function of the edge set: one lookup in the 2^E-bit
      // table built once per handle (2 MB for the 4x4 grid, L2-resident) instead of a divergent flood
      uint32_t bit = 1u << (rv >> 10), g2 = graph & ~bit;
      bool keep = (pg_ldg(&p.conn_table[g2 >> 5]) >> (g2 & 31)) & 1u;
      graph = keep ? g2 : graph;
      cur -= keep ? 2 : 0;
      continue;
    }
    unsigned ab = m.edge_tab[i];
    int a = ab & 255, b = ab >> 8;
    int lo = a < b ? a : b;
    bool horiz = (a > b ? a - b : b - a) == 1 && W != 1;  // on a 1-wide map every edge is vertical (t <-> t + W = t + 1)
    if (horiz) bclr(E, lo); else bclr(S, lo);
    if (still_connected<TMAX>(c, p, E, S, a, b, st, gt)) cur -= 2;
    else { if (horiz) bset(E, lo); else bset(S, lo); }
  }
  }
  if (tabled) {  // back to the boards: E has a hole after every row, S is contiguous
    graph_to_boards(c, graph, E.w[0], S.w[0]);
    m.graph = graph; m.graph_valid = true;
  }
  // map_graph_to_tile_map_object (:269-334); an E bit is only ever set left of the last column
  for (int t = 0; t < T; t++) {
    int ex = 0;
    if (t >= W && bget(S, t - W)) ex |= 1;
    if (bget(E, t)) ex |= 2;
    if (bget(S, t)) ex |= 4;
    if (t > 0 && bget(E, t - 1)) ex |= 8;
    m.tiles[t] = (uint16_t)ex;
  }
  m.tiles[st] |= (uint16_t)(1 << sd);
  m.tiles[gt] |= (uint16_t)(1 << gd);
  // add_connections_to_borders (:337-371): slots in host-table order, default start/goal removed
  if (RNG == PGTG_RNG_PHILOX) {
    const uint64_t chosen = choose_border_slots<RNG, uint64_t>(c, rng);
    for (int i = 0; i < c.n_border_slots; i++)
      if ((chosen >> i) & 1ull) { const unsigned v = m.border_slots[i]; m.tiles[v & 255] |= (uint16_t)(1 << (v >> 8)); }
  } else {
    uint64_t slots = c.n_border_slots >= 64 ? ~0ull : ((1ull << c.n_border_slots) - 1ull);
    int n_slots = c.n_border_slots;
    for (int k = 0; k < c.border_connections && n_slots > 0; k++) {
      int idx = rng.index(PGTG_STREAM_MAP, n_slots);  // :367
      uint32_t lo32 = (uint32_t)slots, hi32 = (uint32_t)(slots >> 32);
      int pc0 = pg_popc(lo32);
      bool hi = idx >= pc0;
      int i = select32(hi ? hi32 : lo32, hi ? idx - pc0 : idx) + (hi ? 32 : 0);
      slots &= ~(1ull << i);
      n_slots--;
      unsigned v = m.border_slots[i];
      m.tiles[v & 255] |= (uint16_t)(1 << (v >> 8));
    }
  }
  // add_obstacles_to_map (:374-472), row-major, one random() per tile whatever the outcome
  if (c.obstacle_probability > 0)
    for (int t = 0; t < T; t++) m.tiles[t] = (uint16_t)(m.tiles[t] | obstacle_draw<RNG>(c, rng, td_exits(m.tiles[t])));
  e.plan = plan_pack(sx, sy, sd, gx, gy, gd, 0);
}

// parse_map_object's path part (parser.py:27-37, 158-164): Dijkstra with unit weights and
// (cost, push counter) keys == FIFO BFS, successors in N, E, S, W insertion order
// (parse_tile_map_to_graph, parser.py:244-276), first-discovered predecessor.
template <int TMAX>
PG_HD void assign_subgoals_bfs(const DevCfg& c, MapView& m, EnvRegs& e) {
  int W = c.W, T = c.T;
  int st = plan_sy(e.plan) * W + plan_sx(e.plan), gt = plan_gy(e.plan) * W + plan_gx(e.plan);
  for (int t = 0; t < T; t++) m.tiles[t] &= 0x07FF;  // clear subgoal dir + used
  m.tiles[gt] |= (uint16_t)((1 + plan_gd(e.plan)) << 11);  // final tile carries the goal direction (parser.py:158)
  int ns = 1;
  bool found = false;
  // a tile has an east / west neighbour iff the full grid has that edge
  auto has_e = [&](int n) { return (c.full_e[n >> 5] >> (n & 31)) & 1u; };
  if (TMAX <= 16) {
    // queue and predecessors as packed nibbles: the whole BFS in registers
    uint64_t q = (uint64_t)st, prev = 0;
    uint32_t seen = 1u << st;
    int qh = 0, qt = 1;
    while (qh < qt) {
      int n = (int)((q >> (4 * qh)) & 15u);
      qh++;
      if (n == gt) { found = true; break; }
      int ex = td_exits(m.tiles[n]);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        int cand = k == 0 ? n - W : k == 1 ? n + 1 : k == 2 ? n + W : n - 1;
        bool ok = k == 0 ? ((ex & 1) && n >= W) : k == 1 ? ((ex & 2) && has_e(n)) : k == 2 ? ((ex & 4) && n + W < T) : ((ex & 8) && n > 0 && has_e(n - 1));
        if (ok && !((seen >> cand) & 1u)) {
          seen |= 1u << cand;
          prev |= (uint64_t)n << (4 * cand);
          q |= (uint64_t)cand << (4 * qt);
          qt++;
        }
      }
    }
    if (found) {
      int cur = gt;
      while (cur != st) {
        int pr = (int)((prev >> (4 * cur)) & 15u);
        int d = cur == pr - W ? 0 : cur == pr + W ? 2 : cur == pr + 1 ? 1 : 3;  // vertical first: on a 1-wide map t + W == t + 1  // find_direction (parser.py:279-306)
        m.tiles[pr] |= (uint16_t)((1 + d) << 11);
        cur = pr; ns++;
      }
    }
  } else {
    uint8_t q[TMAX], prev[TMAX];
    Board<TMAX> seen;
    bzero(seen);
    int qh = 0, qt = 0;
    bset(seen, st); q[qt++] = (uint8_t)st;
    while (qh < qt) {
      int n = q[qh++];
      if (n == gt) { found = true; break; }
      int ex = td_exits(m.tiles[n]);
      int cand[4] = {n - W, n + 1, n + W, n - 1};
      bool ok[4] = {(ex & 1) && n >= W, (ex & 2) && has_e(n), (ex & 4) && n + W < T, (ex & 8) && n > 0 && has_e(n - 1)};
      for (int k = 0; k < 4; k++)
        if (ok[k] && !bget(seen, cand[k])) { bset(seen, cand[k]); prev[cand[k]] = (uint8_t)n; q[qt++] = (uint8_t)cand[k]; }
    }
    if (found) {
      int cur = gt;
      while (cur != st) {
        int pr = prev[cur];
        int d = cur == pr - W ? 0 : cur == pr + W ? 2 : cur == pr + 1 ? 1 : 3;  // vertical first: on a 1-wide map t + W == t + 1
        m.tiles[pr] |= (uint16_t)((1 + d) << 11);
        cur = pr; ns++;
      }
    }
  }
  if (!found) e.err |= 8;
  e.plan = (e.plan & 0xFFFFFu) | (unsigned)ns << 20;
}

// The path is a pure function of the inner edge set when start and goal are fixed: with the
// connectivity table on and T <= 16 it is read from a table built once per handle by running
// assign_subgoals_bfs on every edge set (path_table_entry), 8 bytes per map instead of a BFS.
template <int TMAX, bool TABLED = false>
PG_HD void assign_subgoals(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e) {
  if (TABLED || (TMAX <= 16 && c.path_tab && m.graph_valid)) {
    uint64_t v = pg_ldg(&p.path_table[m.graph]);
    for (int t = 0; t < c.T; t++) m.tiles[t] = (uint16_t)((m.tiles[t] & 0x07FF) | (unsigned)((v >> (3 * t)) & 7u) << 11);
    if (v >> 63) e.err |= 8;
    e.plan = (e.plan & 0xFFFFFu) | (unsigned)((v >> 48) & 0x1FFu) << 20;
    return;
  }
  if (!TABLED) assign_subgoals_bfs<TMAX>(c, m, e);
}

// one entry of the path table: edge set `graph` -> packed subgoal directions (scratch: T descriptors)
PG_HD uint64_t path_table_entry(const DevCfg& c, const Lut& L, uint32_t graph, uint16_t* scratch) {
  uint32_t E, S;
  graph_to_boards(c, graph, E, S);
  for (int t = 0; t < c.T; t++) {
    int ex = 0;
    if (t >= c.W && ((S >> (t - c.W)) & 1u)) ex |= 1;
    if ((E >> t) & 1u) ex |= 2;
    if ((S >> t) & 1u) ex |= 4;
    if (t > 0 && ((E >> (t - 1)) & 1u)) ex |= 8;
    scratch[t] = (uint16_t)ex;
  }
  EnvRegs e;
  e.x = e.y = e.vx = e.vy = 0; e.misc = 0; e.next_car_id = 0; e.err = 0; e.cursor = 0; e.flags = 0; e.elapsed = 0; e.episode = 0;
  e.plan = plan_pack(c.start_x, c.start_y, c.start_dir, c.goal_x, c.goal_y, c.goal_dir, 0);
  MapView m = {c, L, scratch, e.plan, nullptr, nullptr, nullptr, 0u, false};
  assign_subgoals_bfs<16>(c, m, e);
  uint64_t v = 0;
  for (int t = 0; t < c.T; t++) v |= (uint64_t)td_sg(scratch[t]) << (3 * t);
  v |= (uint64_t)((e.plan >> 20) & 0x1FFu) << 48;
  if (e.err & 8) v |= 1ull << 63;
  return v;
}

// plan word bits 29-30: index of the start square among map.starters (map_rng.choice, :635)
PG_HOSTDEV int plan_start_index(unsigned pl) { return (pl >> 29) & 3; }

// The map of one episode: tile descriptors with their subgoal directions, the plan word (start /
// goal / number of subgoals) and the start-square draw -- everything PGTGEnv.reset takes from
// map_rng (environment.py:601-635). It depends only on (seed, episode), never on the actions, so
// it can be built ahead of time by the map-generation kernel.
// POOL = false: the generator alone (the map-generation kernel, which a level set replaces by phase_serve_level).
template <int RNG, int TMAX, bool TABLED = false, bool POOL = true>
PG_HD void build_map(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, Rng<RNG>& rng) {
  if (POOL && RNG == PGTG_RNG_PHILOX && c.num_levels) {  // level set: the pool's map and the level block's start square (phase_serve_level)
    uint32_t w1;
    const uint32_t lv = level_draw(c, p.key[rng.env], e.episode, rng.env, &w1);
    for (int t = 0; t < c.T; t++) m.tiles[t] = pg_ldg(&p.level_tiles[(size_t)lv * c.T + t]);
    e.plan = pg_ldg(&p.level_plan[lv]);
    if (start_line_labelled(m.tiles[plan_sy(e.plan) * c.W + plan_sx(e.plan)], e.plan)) e.plan |= pg_umulhi(w1, 3u) << 29;
    else e.err |= 64;
    m.plan = e.plan;
    return;
  }
  if (!TABLED && c.fixed_map) {
    for (int t = 0; t < c.T; t++) m.tiles[t] = pg_ldg(&p.fixed_tiles[t]);
    e.plan = p.fixed_plan;
  } else {
    generate_map<RNG, TMAX, TABLED>(c, p, m, e, rng);
  }
  assign_subgoals<TMAX, TABLED>(c, p, m, e);
  m.plan = e.plan;
  // self.position = map_rng.choice(self.map.starters) (:635): 3 squares of the start line, x-major
  int stile = m.start_tile(), sd = plan_sd(e.plan);
  unsigned lab = (m.line_labels(stile, m.tiles[stile]) >> (4 * sd)) & 15;
  if (lab == 3) e.plan |= (unsigned)rng.index(PGTG_STREAM_MAP, 3) << 29;
  else e.err |= 64;
  m.plan = e.plan;
}

// build_map for maps that are a function of the surviving edge set and a few draws (Philox, both tables, fixed start / goal,
// 8 or 16 tiles -- the headline configuration and every BASELINE configuration on the default 4x4 grid): the descriptors are
// assembled in registers, two per word, from the edge boards, the border picks and the path-table entry, and stored straight
// to the ring -- no per-tile loops over shared memory, no staged tables. Same bits as build_map (both are tested).
PG_HOSTDEV bool map_in_registers(const DevCfg& c) {
  return c.conn_bits != 0 && c.path_tab && (c.T == 8 || c.T == 16) && c.start_mode == 0 && c.goal_mode == 0 && !c.fixed_map;
}
template <int RNG>
PG_HD void build_map_in_registers(const DevCfg& c, const DevPtrs& p, EnvRegs& e, Rng<RNG>& rng, uint8_t* arr, uint32_t* dst /* T / 2 words, 16-byte aligned */) {
  const uint32_t graph = remove_edges_tabled<RNG>(c, p, rng, arr);
  const uint64_t v = pg_ldg(&p.path_table[graph]);  // 3-bit subgoal direction per tile | ns << 48 | unreachable << 63
  uint32_t E, S;
  graph_to_boards(c, graph, E, S);
  const uint32_t Sn = S << c.W, Ew = E << 1;  // map_graph_to_tile_map_object (:269-334): exits N E S W
  const int st = c.start_y * c.W + c.start_x, gt = c.goal_y * c.W + c.goal_x;
  uint64_t border = (uint64_t)(1u << c.start_dir) << (4 * st) | (uint64_t)(1u << c.goal_dir) << (4 * gt);
  for (uint32_t chosen = choose_border_slots<RNG, uint32_t>(c, rng); chosen != 0u; chosen &= chosen - 1u) {  // <= 32 slots with <= 16 tiles
    const unsigned s = pg_ldg(&p.border_slots[pg_ffs(chosen) - 1]);  // tile | direction << 8
    border |= (uint64_t)(1u << (s >> 8)) << (4 * (s & 255u));
  }
  if (c.obstacle_probability > 0) {
    // obstacles draw tile by tile, a lane-dependent number of words each: a rolled loop, one 32-bit store per tile pair
    for (int k = 0; 2 * k < c.T; k++) {
      uint32_t w = 0;
      for (int h = 0; h < 2; h++) {
        const int t = 2 * k + h;
        const uint32_t ex = ((Sn >> t) & 1u) | ((E >> t) & 1u) << 1 | ((S >> t) & 1u) << 2 | ((Ew >> t) & 1u) << 3 | ((uint32_t)(border >> (4 * t)) & 15u);
        const uint32_t sg = (uint32_t)(v >> (3 * t)) & 7u;
        w |= (ex | obstacle_draw<RNG>(c, rng, (int)ex) | sg << 11) << (16 * h);
      }
      dst[k] = w;
    }
  } else {
    const uint32_t sg_lo = (uint32_t)v, sg_hi = (uint32_t)(v >> 24);  // tiles 0-7 in bits 0-23, tiles 8-15 in bits 24-47
    const uint32_t bd_lo = (uint32_t)border, bd_hi = (uint32_t)(border >> 32);
    uint32_t out[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      uint32_t w = 0;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int t = 2 * k + h;
        const uint32_t ex = ((Sn >> t) & 1u) | ((E >> t) & 1u) << 1 | ((S >> t) & 1u) << 2 | ((Ew >> t) & 1u) << 3 | (((t < 8 ? bd_lo : bd_hi) >> (4 * (t & 7))) & 15u);
        const uint32_t sg = ((t < 8 ? sg_lo : sg_hi) >> (3 * (t & 7))) & 7u;
        w |= (ex | sg << 11) << (16 * h);
      }
      out[k] = w;
    }
    { uint4 q; q.x = out[0]; q.y = out[1]; q.z = out[2]; q.w = out[3]; ((uint4*)dst)[0] = q; }
    if (c.T == 16) { uint4 q; q.x = out[4]; q.y = out[5]; q.z = out[6]; q.w = out[7]; ((uint4*)dst)[1] = q; }
  }
  if (v >> 63) e.err |= 8;
  e.plan = plan_pack(c.start_x, c.start_y, c.start_dir, c.goal_x, c.goal_y, c.goal_dir, 0) | (unsigned)((v >> 48) & 0x1FFu) << 20;
  // self.position = map_rng.choice(self.map.starters) (:635): drawn iff the start line is still labelled "start"
  // (MapView::line_labels: a subgoal label on the same line comes first)
  const uint32_t ex_st = ((Sn >> st) & 1u) | ((E >> st) & 1u) << 1 | ((S >> st) & 1u) << 2 | ((Ew >> st) & 1u) << 3 | (1u << c.start_dir);
  const int sg_st = (int)((v >> (3 * st)) & 7u);
  const bool start_labelled = !(sg_st && st != gt && sg_st - 1 == c.start_dir && ((ex_st >> (sg_st - 1)) & 1u));
  if (start_labelled) e.plan |= (unsigned)rng.index(PGTG_STREAM_MAP, 3) << 29;
  else e.err |= 64;
}

// the rest of PGTGEnv.reset (environment.py:635-656) on a finished map
// (EXT: the warp-parallel traffic tick creates the spawner list and the initial traffic itself)
template <int RNG, bool LEAN = false, bool EXT = false>
PG_HD void begin_episode(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, Rng<RNG>& rng, int env) {
  e.flags |= EF_TILES_DIRTY | EF_RESET;
  int stile = m.start_tile(), sd = plan_sd(e.plan);
  int k = plan_start_index(e.plan);
  int ox = plan_sx(e.plan) * TILE, oy = plan_sy(e.plan) * TILE;
  (void)stile;
  int sq = m.L.line_sq[sd][k < 3 ? k : 0];  // k-th square of the start line, x-major (map.starters order)
  e.x = ox + sq / TILE; e.y = oy + sq % TILE;
  e.vx = e.vy = 0;
  e.misc = 0;  // flat_tire, light counter, cars (:637-650)
  e.next_car_id = 0;
  if (!LEAN && c.vis_words) {
    for (int i = 0; i < c.vis_words; i++) p.visited[(size_t)i * c.N + env] = 0;
    visited_test_set(c, p, env, e.x, e.y, true);  // positions_path = [position] (:643)
  }
  if (RNG == PGTG_RNG_NUMPY) rng.np_begin_episode();  // children 5r+1..5r+4 of this reset (:593-599)
  if (!LEAN && !EXT && c.traffic_density > 0) {  // :652-653
    if (RNG == PGTG_RNG_PHILOX) build_spawner_list_tile_major(c, p, m, env); else build_spawner_list(c, p, m, env);
    int64_t cur; uint32_t err;
    uint32_t r = create_initial_traffic<RNG>(c, p, m, e, env, rng.kcount[PGTG_STREAM_CAR], &cur, &err);
    e.misc = misc_pack(misc_flat(e.misc), misc_light(e.misc), (int)(r & 0xFFFFu), misc_half(e.misc));
    e.next_car_id = r >> 16; e.cursor = cur; e.err |= err;
  }
}

// PGTGEnv.reset (environment.py:581-656), map built in place
template <int RNG, int TMAX, bool EXT = false>
PG_HD void env_reset(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, int env) {
  e.episode++;
  e.elapsed = 0;
  Rng<RNG> rng(p, e, env);
  build_map<RNG, TMAX>(c, p, m, e, rng);
  begin_episode<RNG, false, EXT>(c, p, m, e, rng, env);
}

// the same with the map taken from the pre-generated "next map" of this env
template <int RNG, bool LEAN = false, bool EXT = false>
PG_HD void env_reset_pregenerated(const DevCfg& c, const DevPtrs& p, MapView& m, EnvRegs& e, int env) {
  e.episode++;
  e.elapsed = 0;
  Rng<RNG> rng(p, e, env);
  const size_t slot = e.episode & 1u;  // ring slot of this episode's pre-generated map
  const uint16_t* nt = p.next_tiles + (slot * c.N + (size_t)env) * c.T;
  if ((c.T & 7) == 0) {
    const uint4* g4 = (const uint4*)nt;
    uint32_t* s32 = (uint32_t*)m.tiles;
    for (int k = 0; k < c.T / 8; k++) { uint4 v = g4[k]; s32[4 * k] = v.x; s32[4 * k + 1] = v.y; s32[4 * k + 2] = v.z; s32[4 * k + 3] = v.w; }
  } else {
    for (int t = 0; t < c.T; t++) m.tiles[t] = nt[t];
  }
  e.plan = p.next_plan[slot * c.N + env];
  m.plan = e.plan;
  begin_episode<RNG, LEAN, EXT>(c, p, m, e, rng, env);
}

// ---------------------------------------------------------------------------------------------
// observation (environment.py:1344-1506): planes as bitmaps
// exit lines of a tile whose label (line_labels: 1 subgoal, 2 used subgoal, 3 start, 4 final goal) belongs to `kind`
PG_HD void label_plane(const MapView& m, unsigned lab, int kind, uint32_t out[3]) {
  for (int d = 0; d < 4; d++) {
    unsigned l = (lab >> (4 * d)) & 15;
    bool on = kind == PGTG_CH_GOALS ? (l == 1 || l == 4) : kind == PGTG_CH_SUBGOAL ? l == 1 : kind == PGTG_CH_FINAL_GOAL ? l == 4
            : kind == PGTG_CH_START ? l == 3 : l == 2;
    if (on) { out[0] |= m.L.exit_line[d][0]; out[1] |= m.L.exit_line[d][1]; out[2] |= m.L.exit_line[d][2]; }
  }
}

PG_HD void tile_plane(const DevCfg& c, const MapView& m, int kind, int t, int phase, uint32_t out[3]) {
  out[0] = out[1] = out[2] = 0;
  unsigned td = m.tiles[t];
  int ex = td_exits(td);
  const uint32_t* wall = m.L.wall[ex];
  switch (kind) {
    case PGTG_CH_WALLS: out[0] = wall[0]; out[1] = wall[1]; out[2] = wall[2]; return;
    case PGTG_CH_ICE: case PGTG_CH_BROKEN: case PGTG_CH_SAND: {
      if (td_otype(td) != kind - PGTG_CH_ICE + 1) return;
      const uint32_t* mk = m.L.mask[td_omask(td)];
      out[0] = mk[0] & ~wall[0]; out[1] = mk[1] & ~wall[1]; out[2] = mk[2] & ~wall[2];
      return;
    }
    case PGTG_CH_LIGHT_GREEN: case PGTG_CH_LIGHT_YELLOW: case PGTG_CH_LIGHT_RED: {
      if (td_otype(td) != 4 || phase != kind - PGTG_CH_LIGHT_GREEN) return;
      const uint32_t* mk = m.L.mask[td_omask(td)];
      out[0] = mk[0] & ~wall[0]; out[1] = mk[1] & ~wall[1]; out[2] = mk[2] & ~wall[2];
      return;
    }
    case PGTG_CH_GOALS: case PGTG_CH_SUBGOAL: case PGTG_CH_FINAL_GOAL: case PGTG_CH_START: case PGTG_CH_USED_SUBGOAL: {
      if (!td_sg(td) && t != m.start_tile()) return;
      label_plane(m, m.line_labels(t, td), kind, out);
      return;
    }
    case PGTG_CH_CAR_SPAWNER: spawner_bits(c, m.L, ex, t % c.W, t / c.W, out); return;
    default: return;
  }
}

PG_HD void emit_bits(uint32_t* bits, uint32_t off, uint32_t v) {
  if (!v) return;
  uint32_t s = off & 31;
  pg_atomic_or(&bits[off >> 5], v << s);
  if (s && (v >> (32 - s))) pg_atomic_or(&bits[(off >> 5) + 1], v >> (32 - s));
}

// one column of a sliding-window plane (environment.py:1369-1385, map.py:80-118): bit iy = the square (X, y0 + iy) carries
// `kind`; squares outside the map are walls and nothing else (fill {"wall"}, :1384)
PG_HD uint32_t sliding_column_bits(const DevCfg& c, const MapView& m, int kind, int phase, int X, int y0) {
  uint32_t col = 0;
  if (X < 0 || X >= c.WS) return kind == PGTG_CH_WALLS ? (c.P >= 32 ? 0xFFFFFFFFu : ((1u << c.P) - 1u)) : 0u;
  const int ttx = X / TILE, lx = X - ttx * TILE;
  for (int iy = 0; iy < c.P;) {
    const int Y = y0 + iy;
    if (Y < 0 || Y >= c.HS) { if (kind == PGTG_CH_WALLS) col |= 1u << iy; iy++; continue; }
    const int tty = Y / TILE, ly = Y - tty * TILE;
    uint32_t w[3];
    tile_plane(c, m, kind, tty * c.W + ttx, phase, w);
    const uint32_t c9 = col9(w, lx) >> ly;  // rows ly.. of this tile column
    int cnt = TILE - ly;
    if (cnt > c.P - iy) cnt = c.P - iy;
    col |= (c9 & ((1u << cnt) - 1u)) << iy;
    iy += cnt;
  }
  return col;
}

// The same planes tile by tile instead of column by column (the lean SLIDE tick, one env per thread): the window covers at
// most ceil((P + 8) / 9)^2 tiles; a tile's 81-bit plane of a kind is built ONCE and its columns are cut into the window, and
// a tile that has nothing of the kind (most kinds on most tiles) costs a descriptor test. Same bits as the column loop.
PG_HD void sliding_planes_by_tile(const DevCfg& c, const MapView& m, int phase, int x0, int y0, uint32_t* bits, uint32_t base) {
  const int P = c.P, PP = P * P;
  const int tx_lo = (x0 + 9 * 64) / TILE - 64, tx_hi = (x0 + P - 1 + 9 * 64) / TILE - 64;  // floor division (x0 >= -window_k)
  const int ty_lo = (y0 + 9 * 64) / TILE - 64, ty_hi = (y0 + P - 1 + 9 * 64) / TILE - 64;
  for (int ch = 0; ch < c.C; ch++) {
    const int kind = c.channel_kind[ch];
    if (kind == PGTG_CH_ZERO || kind == PGTG_CH_TRAFFIC) continue;  // (no cars in the lean tick)
    const uint32_t off = base + ch * PP;
    for (int ttx = tx_lo; ttx <= tx_hi; ttx++) {
      const int ix_lo = ttx * TILE - x0 > 0 ? ttx * TILE - x0 : 0, ix_hi = ttx * TILE + TILE - x0 < P ? ttx * TILE + TILE - x0 : P;
      for (int tty = ty_lo; tty <= ty_hi; tty++) {
        const int iy_lo = tty * TILE - y0 > 0 ? tty * TILE - y0 : 0, iy_hi = tty * TILE + TILE - y0 < P ? tty * TILE + TILE - y0 : P;
        const uint32_t rows = (1u << (iy_hi - iy_lo)) - 1u;  // <= 9 rows of this tile
        if (ttx < 0 || ttx >= c.W || tty < 0 || tty >= c.H) {  // outside the map: walls and nothing else (:1384)
          if (kind == PGTG_CH_WALLS)
            for (int ix = ix_lo; ix < ix_hi; ix++) emit_bits(bits, off + ix * P + iy_lo, rows);
          continue;
        }
        uint32_t w[3];
        tile_plane(c, m, kind, tty * c.W + ttx, phase, w);
        if (!(w[0] | w[1] | w[2])) continue;
        const int ly = y0 + iy_lo - tty * TILE;
        for (int ix = ix_lo; ix < ix_hi; ix++) emit_bits(bits, off + ix * P + iy_lo, (col9(w, x0 + ix - ttx * TILE) >> ly) & rows);
      }
    }
  }
}

// writes env's C*P*P observation bits at bit offset `base` of `bits`, plus position/velocity/nsd
// (planes = false: only the scalars -- the caller writes the planes itself, e.g. one window column per thread)
// (SLIDE: the lean instantiation that keeps the sliding window and next_subgoal_direction -- still no cars, no rules)
template <bool LEAN = false, bool SLIDE = false>
PG_HD void env_observe(const DevCfg& c, const DevPtrs& p, const MapView& m, const EnvRegs& e, int env, uint32_t* bits,
                        uint32_t base, int32_t* pos, int32_t* vel, int32_t* nsd, bool planes = true) {
  int pix = e.x < 0 ? 0 : (e.x > c.WS - 1 ? c.WS - 1 : e.x);  // :1352-1356
  int piy = e.y < 0 ? 0 : (e.y > c.HS - 1 ? c.HS - 1 : e.y);
  int tx = pix / TILE, ty = piy / TILE;
  int phase = light_phase(c, misc_light(e.misc));
  const int ncars = LEAN ? 0 : misc_ncars(e.misc);
  const uint64_t* live = LEAN ? nullptr : car_list(c, p, env, misc_half(e.misc));
  int PP = c.P * c.P;
  if (!LEAN && !planes && !c.sliding) {
    pos[0] = pix - tx * TILE; pos[1] = piy - ty * TILE;
  } else if ((LEAN && !SLIDE) || (!c.sliding && c.obs_fast)) {
    // Fixed window, kind by kind: a tile has walls, at most ONE obstacle / light plane, goal-ish
    // lines only on path tiles; everything else stays zero and costs nothing (same bits as the
    // channel loop below, which remains for feature lists that name a kind twice).
    int t = ty * c.W + tx, ch;
    unsigned td = m.tiles[t];
    int ex = td_exits(td);
    const uint32_t* wall = m.L.wall[ex];
    if ((ch = c.kind_channel[PGTG_CH_WALLS]) >= 0) {
      uint32_t off = base + ch * 81;
      emit_bits(bits, off, wall[0]); emit_bits(bits, off + 32, wall[1]); emit_bits(bits, off + 64, wall[2]);
    }
    int ot = td_otype(td);
    if (ot) {
      ch = ot <= 3 ? c.kind_channel[PGTG_CH_ICE + ot - 1] : ot == 4 ? c.kind_channel[PGTG_CH_LIGHT_GREEN + phase] : -1;
      if (ch >= 0) {
        const uint32_t* mk = m.L.mask[td_omask(td)];
        uint32_t off = base + ch * 81;
        emit_bits(bits, off, mk[0] & ~wall[0]); emit_bits(bits, off + 32, mk[1] & ~wall[1]); emit_bits(bits, off + 64, mk[2] & ~wall[2]);
      }
    }
    if (td_sg(td) || t == m.start_tile()) {
      unsigned lab = m.line_labels(t, td);
      for (int kind = PGTG_CH_GOALS; kind <= PGTG_CH_USED_SUBGOAL; kind = kind == PGTG_CH_GOALS ? PGTG_CH_SUBGOAL : kind + 1) {
        if ((ch = c.kind_channel[kind]) < 0) continue;
        uint32_t w[3] = {0u, 0u, 0u};
        label_plane(m, lab, kind, w);
        uint32_t off = base + ch * 81;
        emit_bits(bits, off, w[0]); emit_bits(bits, off + 32, w[1]); emit_bits(bits, off + 64, w[2]);
      }
    }
    if (!LEAN && ncars && (ch = c.kind_channel[PGTG_CH_TRAFFIC]) >= 0) {  // :1397-1409
      uint32_t w[3] = {0u, 0u, 0u};
      for (int k = 0; k < ncars; k++) {
        unsigned xy = car_xy(live[k]);
        int lx = (int)(xy & 255) - tx * TILE, ly = (int)(xy >> 8) - ty * TILE;
        if (lx >= 0 && lx < TILE && ly >= 0 && ly < TILE) or_bit81(w, lx * TILE + ly);
      }
      uint32_t off = base + ch * 81;
      emit_bits(bits, off, w[0]); emit_bits(bits, off + 32, w[1]); emit_bits(bits, off + 64, w[2]);
    }
    if (!LEAN && (ch = c.kind_channel[PGTG_CH_CAR_SPAWNER]) >= 0) {
      uint32_t w[3] = {0u, 0u, 0u};
      spawner_bits(c, m.L, ex, tx, ty, w);
      uint32_t off = base + ch * 81;
      emit_bits(bits, off, w[0]); emit_bits(bits, off + 32, w[1]); emit_bits(bits, off + 64, w[2]);
    }
    pos[0] = pix - tx * TILE; pos[1] = piy - ty * TILE;  // :1448-1461
  } else if (!LEAN && !c.sliding) {  // (the lean predicate asks for obs_fast with the fixed window)
    int t = ty * c.W + tx;
    for (int ch = 0; ch < c.C; ch++) {
      int kind = c.channel_kind[ch];
      uint32_t w[3];
      if (kind == PGTG_CH_TRAFFIC) {  // :1397-1409
        w[0] = w[1] = w[2] = 0;
        for (int k = 0; k < ncars; k++) {
          unsigned xy = car_xy(live[k]);
          int lx = (int)(xy & 255) - tx * TILE, ly = (int)(xy >> 8) - ty * TILE;
          if (lx >= 0 && lx < TILE && ly >= 0 && ly < TILE) or_bit81(w, lx * TILE + ly);
        }
      } else if (kind == PGTG_CH_ZERO) continue;
      else tile_plane(c, m, kind, t, phase, w);
      uint32_t off = base + ch * 81;
      emit_bits(bits, off, w[0]); emit_bits(bits, off + 32, w[1]); emit_bits(bits, off + 64, w[2]);
    }
    pos[0] = pix - tx * TILE; pos[1] = piy - ty * TILE;  // :1448-1461
  } else {
    int k = c.window_k, x0 = e.x - k, y0 = e.y - k;  // window around the UNCLAMPED position (:1370-1377)
    if (LEAN) { if (planes) sliding_planes_by_tile(c, m, phase, x0, y0, bits, base); }
    else
    for (int ch = 0; planes && ch < c.C; ch++) {
      int kind = c.channel_kind[ch];
      if (kind == PGTG_CH_ZERO) continue;
      uint32_t off = base + ch * PP;
      if (kind == PGTG_CH_TRAFFIC) {
        for (int q = 0; q < ncars; q++) {
          unsigned xy = car_xy(live[q]);
          int ix = (int)(xy & 255) - x0, iy = (int)(xy >> 8) - y0;
          if (ix >= 0 && ix < c.P && iy >= 0 && iy < c.P) emit_bits(bits, off + ix * c.P + iy, 1u);
        }
        continue;
      }
      for (int ix = 0; ix < c.P; ix++) emit_bits(bits, off + ix * c.P, sliding_column_bits(c, m, kind, phase, x0 + ix, y0));
    }
    pos[0] = k; pos[1] = k;  // quirk A.3-4
  }
  vel[0] = e.vx; vel[1] = e.vy;
  int d = -1;
  if ((!LEAN || SLIDE) && c.use_nsd) {  // :1466-1504
    int sg = td_sg(m.tiles[ty * c.W + tx]);  // map.py:120-141
    d = sg ? sg - 1 : -1;
    if (d == -1 || c.sliding) {
      int gx, gy;
      if (m.nearest_goal(pix, piy, gx, gy)) {
        int R = c.lut_radius;
        d = (pg_ldg(&p.dirlut[(gy - piy + R) * (2 * R + 1) + (gx - pix + R)]) >> 3) & 7;
      }
    }
  }
  *nsd = d;
}

}  // namespace pgtg
