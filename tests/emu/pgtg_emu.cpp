// pgtg_emu.cpp -- HOST EMULATION of the pgtg_b200 kernel phases. TEST INFRASTRUCTURE ONLY.
//
// Compiles the product's per-env logic (pgtg_b200/csrc/pgtg_logic.cuh, pgtg_phases.cuh) and its
// C-ABI implementation (pgtg_api_impl.hpp) with g++ over a host-memory backend, running the CTA
// phases as plain loops. It exists so that the CPU test-suite (-m "not gpu") can replay the golden
// reference traces through the SAME logic the sm_100a kernels execute, without a GPU. It is never
// loaded by the pgtg_b200 package, bench.py or smoke(): the product has no CPU path.
#include <stdlib.h>
#include <string.h>

#include "../../pgtg_b200/csrc/pgtg_phases.cuh"
#include "../../pgtg_b200/csrc/pgtg_traffic.cuh"

struct pgtg_env;
static void* bk_alloc(size_t n) { void* p = nullptr; if (posix_memalign(&p, 256, n)) return nullptr; return p; }
static void bk_free(void* p) { free(p); }
static int bk_set_device(int) { return 0; }
static int bk_h2d(void* d, const void* s, size_t n, void*) { memcpy(d, s, n); return 0; }
static int bk_d2h(void* d, const void* s, size_t n, void*) { memcpy(d, s, n); return 0; }
static int bk_d2d(void* d, const void* s, size_t n, void*) { memcpy(d, s, n); return 0; }
static void* bk_stream_create() { return malloc(1); }
static void bk_stream_destroy(void* s) { free(s); }
static int bk_memset(void* d, int v, size_t n) { memset(d, v, n); return 0; }
static int bk_memset_async(void* d, int v, size_t n, void*) { memset(d, v, n); return 0; }
static int bk_sync(void*) { return 0; }
// the emulation runs everything in program order: streams and events are no-ops
static int bk_side_create(void** s, void** a, void** b, void** c, int* sms) { *s = *a = *b = *c = nullptr; *sms = 1; return 0; }
static void bk_side_destroy(void*, void*, void*, void*) {}
static int bk_stream_wait(void*, void*) { return 0; }
static const char* bk_error() { return "emu"; }
static int bk_dl_device_type() { return 1; }  // kDLCPU
static void* bk_event_create() { return malloc(1); }
static void bk_event_destroy(void* ev) { free(ev); }
static int bk_event_record(void*, void*) { return 0; }
static double bk_event_elapsed(void*, void*) { return 0.0; }
static int bk_launch(pgtg_env*, int, const uint8_t*, const int64_t*, const void*, int, void*);
static int bk_stats_reduce(pgtg_env*, void*);
static int bk_stats_reset(pgtg_env*, void*);
static int bk_flatten(pgtg_env*, void*);
static int bk_info(pgtg_env*, int32_t*);
static int bk_error_or(pgtg_env*, uint32_t*);
static bool bk_inline_mapgen() { return false; }
static int bk_conn_table_max_bits() { return 13; }  // CPU tests: tables up to 8192 entries (e.g. 3x3 maps)
static int bk_build_conn_table(pgtg_env*, uint32_t*);
static int bk_build_path_table(pgtg_env*, uint64_t*);
// the device's choice between the traffic tick and the general tick; 96 emulated threads: flat loops get several rounds
static void bk_traffic_geometry(const pgtg::DevCfg& c, int* G, int* NT) { const bool fits = pgtg::tk_fits(c, 32); *G = fits ? 32 : 0; *NT = fits ? 96 : 0; }

#include "../../pgtg_b200/csrc/pgtg_api_impl.hpp"

template <int RNG, int TMAX, bool PREGEN, bool LEAN = false, bool SLIDE = false>
static void run_block(pgtg_env* h, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes,
                      int blk, unsigned char* smem) {
  const DevCfg& c = h->dc;
  const DevPtrs& p = h->dp;
  int B = h->block, env0 = blk * B, nvalid = c.N - env0 < B ? c.N - env0 : B;
  BlockShared sh = carve_shared(smem, c, B);
  for (int t = 0; t < B; t++) phase_stage(c, p, sh, t, B, env0, nvalid, true);
  int n_done = 0;
  double st[8] = {0};
  if (mode == MODE_STEP) {
    for (int t = 0; t < nvalid; t++) {
      int env = env0 + t;
      int a = action_bytes == 8 ? (int)((const int64_t*)actions)[env] : ((const int32_t*)actions)[env];
      StepResult r = phase_step<RNG, LEAN>(c, p, sh, t, env, a);
      if (r.outcome) {
        sh.done_list[n_done++] = t;
        st[0] += 1; st[1] += r.ep_return; st[2] += sh.regs[t].elapsed;
        st[3] += r.outcome == 2; st[4] += r.outcome == 1; st[5] += r.outcome == 3;
        if (c.eval_on) { st[6] += r.ep_disc; st[7] += r.ep_disc < 0; }
      }
    }
    if (c.write_final_obs && n_done) {
      for (int k = 0; k < n_done; k++) { if (LEAN) phase_emit<LEAN, SLIDE>(c, p, sh, sh.done_list[k], env0 + sh.done_list[k], true); else phase_emit(c, p, sh, sh.done_list[k], env0 + sh.done_list[k], true); }
      if (LEAN) {  // the lean FINAL instantiation expands the finished envs' rows 32 bytes at a time
        int words[8] = {0};
        for (int k = 0; k < n_done; k++) words[sh.done_list[k] >> 5] |= (int)(1u << (sh.done_list[k] & 31));
        for (int t = 0; t < B; t++) phase_expand_final_vec(c, p.f_obs_map, sh, t, B, env0, nvalid, words);
      } else
      for (int t = 0; t < B; t++) phase_expand_final(c, p.f_obs_map, sh, t, B, env0, n_done);
      for (int i = 0; i < sh.bits_words; i++) sh.bits[i] = 0;
    }
  } else if (mode == MODE_RESET) {
    for (int t = 0; t < nvalid; t++) {
      int env = env0 + t;
      sh.regs[t] = load_regs(c, p, env);
      if (!mask || mask[env]) {
        if (seeds) { p.key[env] = (uint64_t)seeds[env]; sh.regs[t].episode = 0; }
        p.ep_return[env] = 0;
        if (p.ep_disc) p.ep_disc[env] = 0;
        sh.done_list[n_done++] = t;
      }
    }
  } else {
    for (int t = 0; t < nvalid; t++) sh.regs[t] = load_regs(c, p, env0 + t);
  }
  if (mode != MODE_OBSERVE && c.pregen && n_done) {  // queue map requests (same rule as the kernel)
    const int per = mode == MODE_RESET ? 2 : 1;
    uint32_t base = p.regen_count[p.parity];
    p.regen_count[p.parity] += (uint32_t)(n_done * per);
    uint2* q = p.regen_list + (size_t)p.parity * 2 * c.N + base;
    for (int k = 0; k < n_done; k++) {
      int local = sh.done_list[k];
      uint32_t ep = sh.regs[local].episode + 1u;
      uint2 r; r.x = (uint32_t)(env0 + local);
      if (mode == MODE_RESET) { r.y = ep + 1u; q[2 * k] = r; r.y = ep + 2u; q[2 * k + 1] = r; }
      else { r.y = ep + 2u; q[k] = r; }
    }
  }
  for (int k = 0; k < n_done; k++) {
    if (PREGEN && mode == MODE_STEP) phase_reset<RNG, TMAX, true, LEAN>(c, p, sh, sh.done_list[k], env0 + sh.done_list[k]);
    else phase_reset<RNG, TMAX, false>(c, p, sh, sh.done_list[k], env0 + sh.done_list[k]);
  }
  for (int t = 0; t < nvalid; t++) phase_emit<LEAN, SLIDE>(c, p, sh, t, env0 + t, false);
  for (int t = 0; t < B; t++) phase_expand(c, p.obs_map, sh, t, B, env0, nvalid, p.obs_packed);
  for (int k = 0; k < 8; k++) p.stats[k] += st[k];
}

template <int RNG, int TMAX, bool TABLED = false>
static void run_mapgen(pgtg_env* h) {
  const DevCfg& c = h->dc;
  const DevPtrs& p = h->dp;
  const int B = 128;
  size_t bytes = mapgen_shared_bytes(c, B);
  unsigned char* smem = (unsigned char*)bk_alloc(bytes);
  uint32_t count = p.regen_count[p.parity];
  const uint2* list = p.regen_list + (size_t)p.parity * 2 * c.N;
  if (RNG == PGTG_RNG_PHILOX && TABLED && map_in_registers(c) && !getenv("PGTG_NO_MAP_IN_REGISTERS")) {  // as the kernel dispatches
    alignas(4) uint8_t arr[32];
    for (uint32_t i = 0; i < count; i++) phase_pregenerate_in_registers<RNG>(c, p, arr, (int)list[i].x, list[i].y);
    free(smem);
    return;
  }
  for (uint32_t i0 = 0; i0 < count; i0 += B) {
    memset(smem, 0xA5, bytes);
    BlockShared sh = carve_mapgen(smem, c, B);
    for (int t = 0; t < B; t++) stage_tables(c, p, sh, t, B);
    for (int t = 0; t < B && i0 + t < count; t++) phase_pregenerate<RNG, TMAX, TABLED>(c, p, sh, t, (int)list[i0 + t].x, list[i0 + t].y);
  }
  free(smem);
}

// The traffic tick (pgtg_traffic.cu) with its barriers turned into loop boundaries.
template <int TMAX, bool PREGEN>
static void run_traffic_block(pgtg_env* h, const void* actions, int action_bytes, int blk, unsigned char* smem) {
  const DevCfg& c = h->dc;
  const DevPtrs& p = h->dp;
  const TkLayout L = tk_layout(c, h->traffic_G);
  const TkShared sh = tk_carve(smem, L);
  const int G = L.G, NT = h->traffic_NT, env0 = blk * G, nvalid = c.N - env0 < G ? c.N - env0 : G;
  BlockShared bs;
  memset(&bs, 0, sizeof bs);
  bs.lut = sh.lut; bs.spread = sh.spread; bs.tiles = sh.tiles; bs.bits = sh.bits; bs.bits_words = sh.bits_words; bs.done_list = sh.done_list;
  for (int t = 0; t < NT; t++) phase_stage(c, p, bs, t, NT, env0, nvalid, true, false);
  for (int i = 0; i < G * sh.occ_words; i++) sh.occ[i] = 0;
  for (int i = 0; i < 32 * 32; i++) sh.wbits[i] = 0;
  for (int i = 0; i < c.T; i++) tk_stage_tile(c, sh, i);
  for (int g = 0; g < nvalid; g++) {
    int env = env0 + g;
    int a = action_bytes == 8 ? (int)((const int64_t*)actions)[env] : ((const int32_t*)actions)[env];
    tk_stage_env(c, p, sh, g, env, a);
  }
  for (int g = 0; g < nvalid; g++) tk_prefix(sh, sh.off, g, nvalid, false);
  if (c.num_rules > 0) for (int i = 0; i < nvalid * c.T; i++) tk_goal_key(c, sh, i / c.T, i % c.T, false);
  const int total = sh.off[G];
  for (int t = 0; t < NT; t++)
    for (int item = t; item < total; item += NT) { int g = sh.item_g[item]; tk_intent(c, p, sh, g, item - sh.off[g], env0 + g); }
  for (int g = 0; g < nvalid; g++) if (sh.env[g].n_cars > 0) tk_resolve_commit(c, p, sh, g, env0 + g, g & 31);
  int n_done = 0;
  double st[8] = {0};
  for (int g = 0; g < nvalid; g++) {
    StepResult r = tk_agent(c, p, sh, g, env0 + g);
    sh.env[g].ng_key = 0xFFFFFFFFu;
    if (r.outcome) {
      sh.done_list[n_done++] = g;
      st[0] += 1; st[1] += r.ep_return; st[2] += sh.env[g].e.elapsed;
      st[3] += r.outcome == 2; st[4] += r.outcome == 1; st[5] += r.outcome == 3;
      if (c.eval_on) { st[6] += r.ep_disc; st[7] += r.ep_disc < 0; }
      if (PREGEN) {
        uint2 q; q.x = (uint32_t)(env0 + g); q.y = sh.env[g].e.episode + 3u;
        p.regen_list[(size_t)p.parity * 2 * c.N + p.regen_count[p.parity]++] = q;
      }
    }
  }
  if (c.write_final_obs && n_done) {
    for (int item = 0; item < total; item++) {
      int g = sh.item_g[item];
      const TEnv& t = sh.env[g];
      if (t.done) tk_car_bit(c, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, t.e.x, t.e.y, sh.fxy[g * sh.MC + item - sh.off[g]]);
    }
    if (c.use_nsd) for (int i = 0; i < nvalid * c.T; i++) if (sh.env[i / c.T].done) tk_goal_key(c, sh, i / c.T, i % c.T, true);
    if (c.sliding) for (int i = 0; i < nvalid * c.C * c.P; i++) if (sh.env[i / (c.C * c.P)].done) tk_sliding_column(c, sh, i / (c.C * c.P), i % (c.C * c.P));
    for (int k = 0; k < n_done; k++) { tk_emit(c, p, sh, sh.done_list[k], env0 + sh.done_list[k], true); sh.env[sh.done_list[k]].ng_key = 0xFFFFFFFFu; }
    for (int t = 0; t < NT; t++) phase_expand_final(c, p.f_obs_map, bs, t, NT, env0, n_done);
    for (int i = 0; i < sh.bits_words; i++) sh.bits[i] = 0;
  }
  for (int item = 0; item < total; item++) {
    int g = sh.item_g[item];
    const TEnv& t = sh.env[g];
    if (!t.done) tk_car_bit(c, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, t.e.x, t.e.y, sh.fxy[g * sh.MC + item - sh.off[g]]);
  }
  if (n_done) {
    for (int k = 0; k < n_done; k++) tk_reset_map<TMAX, PREGEN>(c, p, sh, sh.done_list[k], env0 + sh.done_list[k]);
    for (int part = 0; part < 3; part++)
      for (int k = 0; k < n_done; k++) tk_reset_traffic(c, p, sh, sh.done_list[k], env0 + sh.done_list[k], 1 << part);
    for (int g = 0; g < nvalid; g++) tk_prefix(sh, sh.off2, g, nvalid, true);
    const int total2 = sh.off2[G];
    for (int t = 0; t < NT; t++)
      for (int item = t; item < total2; item += NT) { int g = sh.item_g[item]; tk_new_car(c, p, sh, g, item - sh.off2[g], env0 + g); }
  }
  if (c.use_nsd) for (int i = 0; i < nvalid * c.T; i++) tk_goal_key(c, sh, i / c.T, i % c.T, true);
  if (c.sliding) for (int i = 0; i < nvalid * c.C * c.P; i++) tk_sliding_column(c, sh, i / (c.C * c.P), i % (c.C * c.P));
  for (int g = 0; g < nvalid; g++) tk_emit(c, p, sh, g, env0 + g, false);
  for (int t = 0; t < NT; t++) phase_expand(c, p.obs_map, bs, t, NT, env0, nvalid, p.obs_packed);
  for (int k = 0; k < 8; k++) p.stats[k] += st[k];
}

static int bk_launch(pgtg_env* h, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void*) {
  int T = h->dc.T;  // same TMAX dispatch as the CUDA backend
  if (mode == MODE_STEP && h->traffic_G > 0) {
    const TkLayout L = tk_layout(h->dc, h->traffic_G);
    unsigned char* smem = (unsigned char*)bk_alloc(L.total);
    int nblk = (h->dc.N + L.G - 1) / L.G;
    for (int b = 0; b < nblk; b++) {
      memset(smem, 0xA5, L.total);
      if (h->dc.pregen) run_traffic_block<16, true>(h, actions, action_bytes, b, smem);
      else if (T <= 16) run_traffic_block<16, false>(h, actions, action_bytes, b, smem);
      else if (T <= 64) run_traffic_block<64, false>(h, actions, action_bytes, b, smem);
      else run_traffic_block<256, false>(h, actions, action_bytes, b, smem);
    }
    free(smem);
    return 0;
  }
  if (mode == MODE_MAPGEN) {
    const bool tabled = h->dc.conn_bits && h->dc.path_tab;  // same dispatch as the CUDA launch code
    if (h->cfg.rng_mode == PGTG_RNG_NUMPY) { if (tabled) run_mapgen<PGTG_RNG_NUMPY, 16, true>(h); else if (T <= 16) run_mapgen<PGTG_RNG_NUMPY, 16>(h); else if (T <= 64) run_mapgen<PGTG_RNG_NUMPY, 64>(h); else run_mapgen<PGTG_RNG_NUMPY, 256>(h); }
    else { if (tabled) run_mapgen<PGTG_RNG_PHILOX, 16, true>(h); else if (T <= 16) run_mapgen<PGTG_RNG_PHILOX, 16>(h); else if (T <= 64) run_mapgen<PGTG_RNG_PHILOX, 64>(h); else run_mapgen<PGTG_RNG_PHILOX, 256>(h); }
    return 0;
  }
  size_t bytes = block_shared_bytes(h->dc, h->block);
  unsigned char* smem = (unsigned char*)bk_alloc(bytes);
  int nblk = (h->dc.N + h->block - 1) / h->block;
  for (int b = 0; b < nblk; b++) {
    memset(smem, 0xA5, bytes);  // shared memory starts undefined on the device too
    bool tape = h->cfg.rng_mode == PGTG_RNG_TAPE;
#define RUN(R, M, G) run_block<R, M, G>(h, mode, mask, seeds, actions, action_bytes, b, smem)
// the lean instantiation is a step-mode specialisation, as in the CUDA launch code
#define RUNL(R, M) do { if (h->dc.lean == 2) run_block<R, M, true, true, true>(h, mode, mask, seeds, actions, action_bytes, b, smem); \
                        else run_block<R, M, true, true>(h, mode, mask, seeds, actions, action_bytes, b, smem); } while (0)
    const bool lean = h->dc.lean && mode == MODE_STEP;
#define RUN3(M) do { bool np = h->cfg.rng_mode == PGTG_RNG_NUMPY; if (tape) RUN(PGTG_RNG_TAPE, M, false); \
    else if (np) { if (h->dc.pregen && lean) RUNL(PGTG_RNG_NUMPY, M); else if (h->dc.pregen) RUN(PGTG_RNG_NUMPY, M, true); else RUN(PGTG_RNG_NUMPY, M, false); } \
    else if (h->dc.pregen && lean) RUNL(PGTG_RNG_PHILOX, M); else if (h->dc.pregen) RUN(PGTG_RNG_PHILOX, M, true); else RUN(PGTG_RNG_PHILOX, M, false); } while (0)
    if (T <= 16) RUN3(16); else if (T <= 64) RUN3(64); else RUN3(256);
#undef RUN3
#undef RUNL
#undef RUN
  }
  free(smem);
  return 0;
}

extern "C" int pgtg_observe(pgtg_env* e, void* stream) {
  if (!e || !e->did_reset) return fail(PGTG_ERR_STATE, "observe before reset");
  bk_launch(e, MODE_OBSERVE, nullptr, nullptr, nullptr, 0, stream);
  e->launches++;
  return PGTG_OK;
}

// the emulation accumulates straight into the 8-double stats buffer
static int bk_stats_reduce(pgtg_env*, void*) { return 0; }
static int bk_stats_reset(pgtg_env* e, void*) { memset(e->dp.stats, 0, 64); return 0; }

static int bk_error_or(pgtg_env* e, uint32_t* out) { uint32_t v = 0; for (int i = 0; i < e->dc.N; i++) v |= e->dp.error[i]; *out = v; return 0; }
static int bk_info(pgtg_env* e, int32_t* out) {
  Lut lut;
  BlockShared sh;
  memset(&sh, 0, sizeof sh);
  sh.lut = &lut;
  for (int t = 0; t < 128; t++) stage_tables(e->dc, e->dp, sh, t, 128, false);
  for (int env = 0; env < e->dc.N; env++) info_env(e->dc, e->dp, lut, env, out);
  return 0;
}

// host loop of the flatten kernel (same index arithmetic)
static int bk_flatten(pgtg_env* e, void*) {
  const DevCfg& c = e->dc;
  const DevPtrs& p = e->dp;
  int dim = e->flat_dim, PP = c.P * c.P, map_dim = c.C * PP, nsd_dim = c.use_nsd ? 9 : 0;
  for (size_t i = 0; i < (size_t)c.N * dim; i++) {
    int env = (int)(i / dim), j = (int)(i - (size_t)env * dim);
    float v;
    if (j < map_dim) { int k = j / PP, cell = j - k * PP; v = (float)p.obs_map[((size_t)env * c.C + e->flat_order[k]) * PP + cell]; }
    else if (j < map_dim + nsd_dim) v = (p.obs_nsd[env] + 1 == j - map_dim) ? 1.0f : 0.0f;
    else if (j < map_dim + nsd_dim + 18) { int q = j - map_dim - nsd_dim; v = (p.obs_position[2 * env + (q >= 9)] == (q >= 9 ? q - 9 : q)) ? 1.0f : 0.0f; }
    else v = (float)p.obs_velocity[2 * env + (j - map_dim - nsd_dim - 18)];
    e->flat[i] = v;
  }
  return 0;
}

// host loop of the path-table builder
static int bk_build_path_table(pgtg_env* e, uint64_t* table) {
  const DevCfg& c = e->dc;
  std::vector<uint16_t> scratch(c.T + 8);
  Lut lut;
  memset(&lut, 0, sizeof(lut));
  for (uint32_t g = 0; g < (1u << c.conn_bits); g++) table[g] = path_table_entry(c, lut, g, scratch.data());
  return 0;
}

// host loop of the connectivity-table builder (same index arithmetic as the kernel)
static int bk_build_conn_table(pgtg_env* e, uint32_t* table) {
  const DevCfg& c = e->dc;
  int s = c.start_y * c.W + c.start_x, g = c.goal_y * c.W + c.goal_x;
  uint32_t total = 1u << c.conn_bits, rowmask = (1u << (c.W - 1)) - 1u, emask = (1u << c.conn_ne) - 1u;
  for (uint32_t w = 0; w < total / 32 + 1; w++) table[w] = 0;
  for (uint32_t idx = 0; idx < total; idx++) {
    uint32_t ec = idx & emask, so = idx >> c.conn_ne, ed = 0;
    for (int r = 0; r < c.H; r++) ed |= ((ec >> (r * (c.W - 1))) & rowmask) << (r * c.W);
    if (flood_connected32(c.W, ed, so, s, g)) table[idx >> 5] |= 1u << (idx & 31);
  }
  return 0;
}
