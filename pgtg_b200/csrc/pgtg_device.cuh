// pgtg_device.cuh -- device-side data layout and per-env logic of the batched PGTG simulator.
//
// Design (B200-first, see DESIGN.md):
//  * env state is structure-of-arrays in HBM; one env per thread for the sequential game logic;
//  * a map is never materialised as squares: every square feature is a pure function of a 16-bit
//    tile descriptor + 81-bit LUT bitmaps staged in shared memory (SURVEY.md A.2);
//  * done envs are compacted per CTA (ballot + scan) and regenerated on device in the same launch;
//  * observations leave the SM as one contiguous, 16-byte-vectorised byte stream per CTA, expanded
//    from a packed bitstring assembled in shared memory.
//
// Reference citations are paths under /root/reference/pgtg/.
#pragma once
#include <stdint.h>
#include <stdlib.h>

// The per-env logic in this header and in pgtg_logic.cuh is written once and compiled twice:
// by nvcc for sm_100a (the product), and by g++ for tests/emu (a host-side emulation of the same
// kernel phases used ONLY by the CPU test-suite to debug the logic without a GPU; the product
// library contains no CPU step path).
#ifdef __CUDACC__
#include <cuda_runtime.h>
#define PG_HD __device__ __forceinline__
#define PG_HDN static __device__ __noinline__
#define PG_HOSTDEV __host__ __device__ inline
#define PG_MEMBER __device__
#define PG_DEVCONST __device__ const
#define pg_umulhi(a, b) __umulhi((a), (b))
#define pg_ffs(v) __ffs((int)(v))
#define pg_popc(v) __popc((unsigned)(v))
#define pg_clz(v) __clz((int)(v))
#define pg_popcll(v) __popcll((unsigned long long)(v))
#define pg_ldg(p) __ldg(p)
#define pg_dmul(a, b) __dmul_rn((a), (b))
#define pg_dadd(a, b) __dadd_rn((a), (b))
#define pg_ddiv(a, b) __ddiv_rn((a), (b))
#define pg_atomic_or(p, v) atomicOr((p), (v))
#define pg_atomic_add(p, v) atomicAdd((p), (v))
#define pg_atomic_cas(p, o, n) atomicCAS((p), (o), (n))
#define pg_atomic_min(p, v) atomicMin((p), (v))
#define pg_store_streaming(ptr, v) __stcs((ptr), (v))  /* written once, never re-read by the kernel: evict-first */
#define pg_prefetch_l2(ptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr))  /* fire-and-forget */
/* 32 bytes with one 256-bit streaming store (sm_100: STG.256); ptr 32-byte aligned */
__device__ __forceinline__ void pg_store_streaming32(void* ptr, uint2 a, uint2 b, uint2 c2, uint2 d) {
  asm volatile("st.global.cs.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(ptr), "r"(a.x), "r"(a.y), "r"(b.x), "r"(b.y), "r"(c2.x), "r"(c2.y), "r"(d.x), "r"(d.y) : "memory");
}
#else
#include <math.h>
#include <string.h>
#define PG_HD static inline
#define PG_HDN static
#define PG_HOSTDEV static inline
#define PG_MEMBER
#define PG_DEVCONST static const
static inline uint32_t pg_umulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
#define pg_ffs(v) __builtin_ffs((int)(v))
#define pg_popc(v) __builtin_popcount((unsigned)(v))
#define pg_clz(v) ((v) ? __builtin_clz((unsigned)(v)) : 32)
#define pg_popcll(v) __builtin_popcountll((unsigned long long)(v))
#define pg_ldg(p) (*(p))
// the emulation build uses -ffp-contract=off, so plain operators are correctly rounded, unfused
#define pg_dmul(a, b) ((a) * (b))
#define pg_dadd(a, b) ((a) + (b))
#define pg_ddiv(a, b) ((a) / (b))
#define pg_atomic_or(p, v) (*(p) |= (v))
static inline uint32_t pg_atomic_add(uint32_t* p, uint32_t v) { uint32_t o = *p; *p = o + v; return o; }
static inline int pg_atomic_add(int* p, int v) { int o = *p; *p = o + v; return o; }
static inline uint32_t pg_atomic_min(uint32_t* p, uint32_t v) { uint32_t o = *p; if (v < o) *p = v; return o; }
static inline uint32_t pg_atomic_cas(uint32_t* p, uint32_t o, uint32_t n) { uint32_t c = *p; if (c == o) *p = n; return c; }
#define pg_store_streaming(ptr, v) (*(ptr) = (v))
#define pg_prefetch_l2(ptr) ((void)(ptr))
struct short4 { short x, y, z, w; };
struct int2 { int x, y; };
struct int4 { int x, y, z, w; };
struct uint4 { unsigned x, y, z, w; };
struct uint2 { unsigned x, y; };
static inline void pg_store_streaming32(void* ptr, uint2 a, uint2 b, uint2 c2, uint2 d) {
  uint2* q = (uint2*)ptr; q[0] = a; q[1] = b; q[2] = c2; q[3] = d;
}
#endif

#include "../../include/pgtg_b200.h"
#include "pgtg_tables.h"

// Warp-collective phases, written once for both builds. On the device the function body runs on every lane of a
// warp (`l` = the lane), PG_FOR_LANES is empty and a per-lane variable is a register; the emulation runs the 32 lanes
// of the warp as a loop around each per-lane block and keeps per-lane variables as arrays. Lanes exchange data only
// through the collectives below or through shared memory, and collectives stand between per-lane blocks.
#ifdef __CUDACC__
#define PG_WARP_LANE const int l = (int)(threadIdx.x & 31u);
#define PG_FOR_LANES
#define PG_LV(type, name) type name
#define LV(name) name
#define PG_BALLOT(out, pred) out = __ballot_sync(0xffffffffu, (pred))
#define PG_REDUCE_OR(out, expr) out = __reduce_or_sync(0xffffffffu, (uint32_t)(expr))
#define PG_MATCH_ANY(name, expr) name = __match_any_sync(0xffffffffu, (uint32_t)(expr))
#define PG_SYNCWARP() __syncwarp()
#else
#define PG_WARP_LANE
#define PG_FOR_LANES for (int l = 0; l < 32; l++)
#define PG_LV(type, name) type name[32]
#define LV(name) name[l]
#define PG_BALLOT(out, pred) { out = 0; for (int l = 0; l < 32; l++) if (pred) out |= 1u << l; }
#define PG_REDUCE_OR(out, expr) { out = 0; for (int l = 0; l < 32; l++) out |= (uint32_t)(expr); }
#define PG_MATCH_ANY(name, expr) { uint32_t k_[32]; for (int l = 0; l < 32; l++) k_[l] = (uint32_t)(expr); \
    for (int l = 0; l < 32; l++) { uint32_t m_ = 0; for (int q = 0; q < 32; q++) if (k_[q] == k_[l]) m_ |= 1u << q; name[l] = m_; } }
#define PG_SYNCWARP()
#endif

namespace pgtg {

constexpr int TILE = 9;
constexpr int MAX_EDGE_TAB = 4 * PGTG_MAX_TILES;  // directed grid edges
constexpr int MAX_BORDER_SLOTS = 64;

// tile descriptor (uint16): exits 0-3 | obstacle type 4-6 | mask id 7-10 | subgoal dir 11-13
// (0 none, 1+dir; on the goal tile 1+goal_dir) | bit 14: subgoal of this tile consumed
constexpr unsigned TD_USED = 1u << 14;
PG_HOSTDEV int td_exits(unsigned td) { return td & 15; }
PG_HOSTDEV int td_otype(unsigned td) { return (td >> 4) & 7; }
PG_HOSTDEV int td_omask(unsigned td) { return (td >> 7) & 15; }
PG_HOSTDEV int td_sg(unsigned td) { return (td >> 11) & 7; }

// plan word: sx 0-3 | sy 4-7 | sdir 8-9 | gx 10-13 | gy 14-17 | gdir 18-19 | num_subgoals 20-28
PG_HOSTDEV unsigned plan_pack(int sx, int sy, int sd, int gx, int gy, int gd, int ns) {
  return (unsigned)sx | (unsigned)sy << 4 | (unsigned)sd << 8 | (unsigned)gx << 10 | (unsigned)gy << 14 |
         (unsigned)gd << 18 | (unsigned)ns << 20;
}
PG_HOSTDEV int plan_sx(unsigned p) { return p & 15; }
PG_HOSTDEV int plan_sy(unsigned p) { return (p >> 4) & 15; }
PG_HOSTDEV int plan_sd(unsigned p) { return (p >> 8) & 3; }
PG_HOSTDEV int plan_gx(unsigned p) { return (p >> 10) & 15; }
PG_HOSTDEV int plan_gy(unsigned p) { return (p >> 14) & 15; }
PG_HOSTDEV int plan_gd(unsigned p) { return (p >> 18) & 3; }
PG_HOSTDEV int plan_ns(unsigned p) { return (p >> 20) & 511; }

// car record (uint64): x 0-7 | y 8-15 | route 16-20 | profile 21-23 | delay 24-25 |
// patience 26-39 (saturating) | id 40-63
constexpr unsigned PATIENCE_MAX = (1u << 14) - 1;
struct Car {
  int x, y, route, profile, delay, patience;
  unsigned id;
};
PG_HOSTDEV uint64_t car_pack(const Car& c) {
  unsigned pat = c.patience > (int)PATIENCE_MAX ? PATIENCE_MAX : (unsigned)c.patience;
  return (uint64_t)(unsigned)c.x | (uint64_t)(unsigned)c.y << 8 | (uint64_t)c.route << 16 | (uint64_t)c.profile << 21 |
         (uint64_t)c.delay << 24 | (uint64_t)pat << 26 | (uint64_t)(c.id & 0xFFFFFFu) << 40;
}
PG_HOSTDEV Car car_unpack(uint64_t v) {
  Car c;
  c.x = (int)(v & 255); c.y = (int)((v >> 8) & 255); c.route = (int)((v >> 16) & 31); c.profile = (int)((v >> 21) & 7);
  c.delay = (int)((v >> 24) & 3); c.patience = (int)((v >> 26) & PATIENCE_MAX); c.id = (unsigned)(v >> 40);
  return c;
}
PG_HOSTDEV unsigned car_xy(uint64_t v) { return (unsigned)(v & 0xFFFF); }

// Values of the config the kernels read; passed by value as a __grid_constant__ kernel parameter
// (constant bank, uniform access).
struct DevCfg {
  int N, W, H, T, WS, HS;  // envs, tiles, squares
  int C, P, sliding, window_k, use_nsd;
  int channel_kind[PGTG_MAX_CHANNELS];
  int kind_channel[16];          // kind -> its channel (-1: not observed); valid when obs_fast
  int lean;                     // plain configuration: the tick runs the LEAN instantiation (see env_step); 2 = its SLIDE variant (sliding window / nsd)
  int obs_fast;                 // fixed window and no kind listed twice: the observation is written kind by kind
  int fixed_map, edges_to_keep, n_edge_tab, border_connections, n_border_slots;
  int start_mode, goal_mode, start_x, start_y, start_dir, goal_x, goal_y, goal_dir, min_sg_dist;
  double obstacle_probability, obstacle_cdf[4];
  double sum_subgoals_reward, final_goal_bonus, crash_penalty, light_penalty, standing_penalty, visited_penalty;
  double ice_p, broken_p, sand_p, traffic_density;
  int light_green, light_yellow, light_total, ignore_traffic_collisions;
  double profile_cdf[5], drv_yellow_stop[5], drv_red_violation[5], drv_patience_threshold[5], drv_push_probability[5],
      drv_speed_multiplier[5], drv_reaction_delay[5];
  int drv_min_following[5];
  int separate_reward_cost, num_rules, max_episode_steps, write_final_obs, max_cars, lut_radius;
  int pregen;  // maps of the next episode are built ahead of time by the map-generation kernel
  int rules_without_traffic;  // some rule has min_traffic <= 0 and min_matching_traffic <= 0
  int tile_stride;   // uint16 elements per env in the shared-memory tile stage (odd word count)
  int vis_w, vis_words;  // visited bitmap geometry (0 when the penalty is off)
  int occ_words, spawner_cap;  // traffic helpers (0 without traffic)
  int obs_bits;      // C * P * P
  uint32_t full_e[8], full_s[8];  // full grid graph: bit t = edge t<->t+1 / t<->t+W exists
  // start-goal connectivity table (procedural maps with fixed start/goal and <= 24 grid edges):
  // bit [compress(E) | S << conn_ne] = start and goal connected in the subgraph (E, S)
  int conn_bits, conn_ne;
  int path_tab;                 // 1: subgoal paths come from DevPtrs.path_table (T <= 16, same index as conn_table)
  int eval_on, gamma_len;        // evaluator statistics (pgtg_set_evaluation): discounted returns with DevPtrs.gamma_pow
  int64_t env_id_base;
  uint64_t seed;
  // level sets (pgtg_config): pool size M (0 = off), sampling (1 = level (env_id_base + env) mod M), first key of the pool.
  // Three ints + padding = 16 bytes: the DevPtrs parameter behind this struct keeps its 16-byte alignment, so kernels that
  // do not use levels keep their parameter loads (and the lean ticks their exact code).
  int num_levels, level_sampling, start_level;
};

// numpy mode: one PCG64 stream (pgtg_device.cuh, 'numpy-exact generator')
struct PcgState {
  uint64_t st_lo, st_hi, inc_lo, inc_hi;
  uint32_t buf, has;  // PCG64's buffered upper half of the last 64-bit output (next_uint32)
};

struct Lut;

// Device pointers (all owned by the handle).
struct DevPtrs {
  // state, SoA
  short4* agent;        // [N] x, y, vx, vy
  uint32_t* misc;       // [N] flat_tire | light_counter << 1 | live car-list half << 15 | n_cars << 16
  uint32_t* elapsed;    // [N]
  uint32_t* episode;    // [N]
  uint32_t* next_car_id;  // [N]
  uint32_t* plan;       // [N]
  uint16_t* tiles;      // [N][T]
  // pregen mode: a ring of two pre-generated maps per env; slot (k & 1) holds the map of episode k
  uint16_t* next_tiles; // [2][N][T]
  uint32_t* next_plan;  // [2][N]
  // map requests (env, episode), double-buffered by launch parity
  uint2* regen_list;    // [2][2N]
  uint32_t* regen_count; // [2]
  int parity;           // launch index & 1: this launch appends to queue `parity`
  uint64_t* cars;       // [N][2][max_cars]: two halves per env, misc bit 15 says which one is live (the other is the
                        // warp-parallel tick's write target / the sequential tick's respawn scratch)
  uint32_t* visited;    // [vis_words][N] or null
  // traffic helpers (allocated when traffic_density > 0)
  uint32_t* occ;        // [occ_words][N] per-tick 2-bit car counters per square (cell x*HS+y), 3 = saturated
  uint16_t* spawners;   // [N][spawner_cap] car_spawner squares in x-major order (x | y << 8), built at reset
  uint16_t* spawner_count;  // [N]
  uint64_t* key;        // [N] philox key / numpy entropy (the env's seed)
  PcgState* pcg;        // [4][pcg_stride] numpy mode: car, ice, broken road, sand PCG64 streams
  size_t pcg_stride;
  int64_t* cursor;      // [N] tape cursor
  int64_t* tape_end;    // [N]
  const double* tape_values;
  const uint8_t* tape_tags;
  uint32_t* error;      // [N] sticky
  double* ep_return;    // [N]
  double* ep_disc;      // [N] running discounted return of the episode (evaluator statistics), or null
  const double* gamma_pow;  // [gamma_len] pow(gamma, t) evaluated on the host
  // tables
  const uint16_t* fixed_tiles;  // [T] (fixed map)
  uint32_t fixed_plan;
  const uint16_t* edge_tab;     // [n_edge_tab] a | b << 8  (edges() order)
  const uint16_t* edge_rev;     // [n_edge_tab] index of the reverse edge | connectivity-table bit of the edge << 10
  const uint16_t* border_slots; // [n_border_slots] tile | dir << 8
  const uint8_t* dirlut;        // (2R+1)^2
  const uint32_t* conn_table;   // [2^conn_bits / 32] or null
  const Lut* lut;               // the LUTs with their derived fields, built once per handle
  const uint8_t* target_lut;    // [16][81][20] per (tile type, local square, route): bit d = the square carries a lane of that route with
                                // direction d, bit 4 + d = it carries 'car_lane all d' (a move INTO it from another tile, :915-932)
  const uint8_t* step_lut;      // [16][81][20] per (tile type, local square, route): bit d = the neighbour square in direction d lies in
                                // the same tile and carries a lane of that route with direction d (bits 4-7: ... carries 'all d')
  const uint64_t* path_table;   // [2^conn_bits] or null: 3-bit subgoal direction of every tile | ns << 48 | unreachable << 63
  const uint2* face_tab;        // [conn_bits] or null: per grid edge, the other three edges of its two grid faces as edge-set masks (bit 31 = no such face)
  const pgtg_rule* rules;
  // outputs
  uint32_t* obs_packed;  // [ceil(N * obs_bits / 32)] the observation planes as bits (env i at bit i * obs_bits), or null
                         // (allocated by the bits observation format, or by the first host-buffer step with bits)
  int8_t* obs_map; int32_t* obs_position; int32_t* obs_velocity; int32_t* obs_nsd;
  double* reward; double* cost; uint8_t* terminated; uint8_t* truncated;
  int32_t* step_state; uint8_t* step_flags;
  int8_t* f_obs_map; int32_t* f_obs_position; int32_t* f_obs_velocity; int32_t* f_obs_nsd;
  double* stats;
  // level sets: the pool, built once by pgtg_create (configuration, not state)
  uint16_t* level_tiles;  // [M][T] descriptors, no subgoal consumed
  uint32_t* level_plan;   // [M] plan words, start-square bits clear
  // the bits observation format (pgtg_set_obs_format): obs_map and f_obs_map are null, the ticks store the planes only as bits,
  // to obs_packed and (terminal observations) here, same layout
  uint32_t* f_obs_packed;
};

// ---------------------------------------------------------------------------------------------
// LUTs (generated from the reference's tile data by tools/gen_tables.py), staged in shared memory
struct Lut {
  uint32_t wall[16][3];
  uint32_t exit_line[4][3];
  uint32_t mask[PGTG_NUM_MASKS][3];
  uint32_t lane_any[16][3];
  uint8_t native_spawner[16];
  uint8_t entry_sq[4];
  // derived once per handle on the host (derive_lut, pgtg_api_impl.hpp):
  uint32_t spawner_cols;  // local columns that can hold a car_spawner
  uint32_t exit_any[3];   // union of the four exit lines
  uint8_t line_sq[4][4];  // the three squares of each exit line in ascending order
  uint8_t line_xy[4][4];  // the same as local x | y << 4
  uint8_t lane_count[16]; // lane squares of a tile type
  uint8_t entry_ok[16];   // per tile type, bit k: the border spawner of slot k + 1 exists (spawner slots, pgtg_logic.cuh)
};
struct LutInit { uint32_t wall[16][3], exit_line[4][3], mask[PGTG_NUM_MASKS][3], lane_any[16][3]; uint8_t native_spawner[16], entry_sq[4]; };
PG_DEVCONST uint64_t g_lane_desc[16][81] = PGTG_TAB_LANE_DESC;

PG_HD bool bit81(const uint32_t* w, int sq) { return (w[sq >> 5] >> (sq & 31)) & 1u; }
PG_HD uint64_t lane_desc(int type, int sq) { return pg_ldg(&g_lane_desc[type][sq]); }
PG_HD int ld_all(uint64_t d) { return (int)(d & 7); }          // 0 none, 1 + dir
PG_HD int ld_n(uint64_t d) { return (int)((d >> 3) & 7); }
PG_HD int ld_route(uint64_t d, int i) { return (int)((d >> (6 + 7 * i)) & 31); }
PG_HD int ld_dir(uint64_t d, int i) { return (int)((d >> (11 + 7 * i)) & 3); }

// square feature bits
enum : unsigned { SF_WALL = 1, SF_SUBGOAL = 2, SF_USED = 4, SF_START = 8, SF_FINAL = 16, SF_ICE = 32, SF_BROKEN = 64, SF_SAND = 128, SF_LIGHT = 256 };

// ---------------------------------------------------------------------------------------------
// Per-env working set. Lives in registers of the thread that currently works on the env and is
// parked in shared memory between the step, reset and observe phases (a different thread of the
// CTA may run the reset of a done env after compaction).
struct EnvRegs {
  int x, y, vx, vy;
  uint32_t misc;  // flat | light << 1 | half << 15 | ncars << 16
  uint32_t elapsed, episode, next_car_id, plan;
  uint32_t err;
  int64_t cursor;
  uint32_t flags;  // bit0 tiles dirty, bit1 done, bit2 plan dirty
};
constexpr uint32_t EF_TILES_DIRTY = 1, EF_DONE = 2, EF_RESET = 4;

// misc word: flat tire 0 | traffic-light counter 1-14 | live half of the env's car list 15 | number of cars 16-31
PG_HOSTDEV int misc_flat(uint32_t m) { return m & 1; }
PG_HOSTDEV int misc_light(uint32_t m) { return (m >> 1) & 0x3FFF; }
PG_HOSTDEV int misc_half(uint32_t m) { return (m >> 15) & 1; }
PG_HOSTDEV int misc_ncars(uint32_t m) { return m >> 16; }
PG_HOSTDEV uint32_t misc_pack(int flat, int light, int ncars, int half = 0) { return (uint32_t)flat | (uint32_t)light << 1 | (uint32_t)half << 15 | (uint32_t)ncars << 16; }

// ---------------------------------------------------------------------------------------------
// Random draws (semantic API shared with the oracle, include/pgtg_b200.h):
//   tape   : draws recorded from the reference's five np_random children (environment.py:593-599)
//   philox : Philox4x32-10, key = env seed, counter = (k, tick, episode, stream)
#ifndef PG_PHILOX_ATTR
#define PG_PHILOX_ATTR PG_HD
#endif
PG_PHILOX_ATTR void philox4x32_10(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t h0 = pg_umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = pg_umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// ---- numpy-exact generator (PGTG_RNG_NUMPY) ----------------------------------------------------------
// Restates, for exactly the calls the reference makes, numpy's SeedSequence (hash pool, spawn keys,
// generate_state), PCG64 (128-bit LCG, XSL-RR output, the buffered 32-bit half) and the Generator
// methods random(), integers()/choice(n) (Lemire's 32-bit rejection), choice(p=...) (cdf +
// searchsorted) and choice(n, k, replace=False) (Floyd's sampling + shuffle), so that SEEDS ALONE
// reproduce the reference: env = Generator(PCG64(SeedSequence(seed))) (gymnasium 0.28.1 seeding),
// reset number r spawns children 5r..5r+4 = map, car, ice, broken road, sand streams
// (environment.py:593-599). Pinned against numpy itself in tests/test_numpy_rng.py.
typedef unsigned __int128 pg_u128;
PG_HD uint32_t ss_hashmix(uint32_t v, uint32_t& hc) { v ^= hc; hc *= 0x931e8875u; v *= hc; v ^= v >> 16; return v; }
PG_HD uint32_t ss_mix(uint32_t x, uint32_t y) { uint32_t r = 0xca01f9ddu * x - 0x4973f715u * y; r ^= r >> 16; return r; }
// PCG64 seeded by SeedSequence(entropy = seed, spawn_key = (child,)): the child streams of one reset
PG_HD void pcg_seed_child(uint64_t seed, uint32_t child, PcgState& s) {
  uint32_t ent[5] = {(uint32_t)seed, (uint32_t)(seed >> 32), 0u, 0u, child};  // run entropy padded to the pool, then the spawn key
  uint32_t pool[4], hc = 0x43b0d7e5u;
#pragma unroll
  for (int i = 0; i < 4; i++) pool[i] = ss_hashmix(ent[i], hc);
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++)
      if (a != b) pool[b] = ss_mix(pool[b], ss_hashmix(pool[a], hc));
#pragma unroll
  for (int b = 0; b < 4; b++) pool[b] = ss_mix(pool[b], ss_hashmix(ent[4], hc));
  uint32_t w[8], hb = 0x8b51f9ddu;  // generate_state(4, uint64)
#pragma unroll
  for (int i = 0; i < 8; i++) { uint32_t v = pool[i & 3] ^ hb; hb *= 0x58f38dedu; v *= hb; v ^= v >> 16; w[i] = v; }
  pg_u128 initstate = ((pg_u128)((uint64_t)w[0] | (uint64_t)w[1] << 32) << 64) | ((uint64_t)w[2] | (uint64_t)w[3] << 32);
  pg_u128 initseq = ((pg_u128)((uint64_t)w[4] | (uint64_t)w[5] << 32) << 64) | ((uint64_t)w[6] | (uint64_t)w[7] << 32);
  const pg_u128 mult = ((pg_u128)0x2360ED051FC65DA4ull << 64) | 0x4385DF649FCCF645ull;
  pg_u128 inc = (initseq << 1) | 1u, st = 0;
  st = st * mult + inc;  // pcg_setseq_128_srandom_r
  st += initstate;
  st = st * mult + inc;
  s.st_lo = (uint64_t)st; s.st_hi = (uint64_t)(st >> 64); s.inc_lo = (uint64_t)inc; s.inc_hi = (uint64_t)(inc >> 64);
  s.buf = 0; s.has = 0;
}
PG_HD uint64_t pcg_next64(PcgState& s) {
  const pg_u128 mult = ((pg_u128)0x2360ED051FC65DA4ull << 64) | 0x4385DF649FCCF645ull;
  pg_u128 st = ((pg_u128)s.st_hi << 64) | s.st_lo, inc = ((pg_u128)s.inc_hi << 64) | s.inc_lo;
  st = st * mult + inc;
  s.st_lo = (uint64_t)st; s.st_hi = (uint64_t)(st >> 64);
  uint64_t x = s.st_hi ^ s.st_lo;
  unsigned r = (unsigned)(s.st_hi >> 58);
  return (x >> r) | (x << ((64u - r) & 63u));
}
PG_HD uint32_t pcg_next32(PcgState& s) {
  if (s.has) { s.has = 0; return s.buf; }
  uint64_t n = pcg_next64(s);
  s.has = 1; s.buf = (uint32_t)(n >> 32);
  return (uint32_t)n;
}
// random_bounded_uint64(0, rng) for rng < 2^32 - 1: Lemire's method on 32-bit draws, inclusive bound
PG_HD uint32_t pcg_bounded(PcgState& s, uint32_t rng) {
  if (rng == 0) return 0;
  uint32_t ex = rng + 1u;
  uint64_t m = (uint64_t)pcg_next32(s) * ex;
  uint32_t left = (uint32_t)m;
  if (left < ex) {
    uint32_t thr = (0u - ex) % ex;
    while (left < thr) { m = (uint64_t)pcg_next32(s) * ex; left = (uint32_t)m; }
  }
  return (uint32_t)(m >> 32);
}

// Philox CAR stream (specification shared with the oracle; the reference's car_rng order is only
// reproduced in the tape / numpy modes). Every car owns one block sequence per tick, so that its draws do
// not depend on how many words the cars before it consumed and 32 cars can draw at once:
//   block b of car slot s at (tick, episode) = philox(counter = (b, tick, episode, STREAM_CAR | (s + 1) << 8), key)
// with s = the car's index in the list when the tick starts, and FIXED word meanings (CW_*). A car-stream
// uniform is one word scaled by 2^-32; an index draw is (word * n) >> 32; one-element choices draw nothing.
// Initial traffic (tick 0 of the episode): car slot j takes lane square perm(j) of the x-major list, perm = a
// 4-round Feistel permutation of [0, 2^m) keyed by the block of slot -1 (field 0), cycle-walked into [0, n);
// its profile and route come from words CW0_* of its own block.
enum { CW_DELAY = 0, CW_SPEED = 1, CW_IDX = 2 /* reaction delay length, or the route drawn on tile entry */, CW_PUSH = 3,
       CW_LIGHT = 4, CW_SPAWNER = 5, CW_SPAWN_ROUTE = 6, CW_PROFILE = 7, CW0_PROFILE = 0, CW0_ROUTE = 1 };
PG_HD void philox_car_block(uint64_t key, uint32_t tick, uint32_t episode, int slot, uint32_t blk, uint32_t w[4]) {
  w[0] = blk; w[1] = tick; w[2] = episode; w[3] = (uint32_t)PGTG_STREAM_CAR | (uint32_t)(slot + 1) << 8;
  philox4x32_10(w[0], w[1], w[2], w[3], (uint32_t)key, (uint32_t)(key >> 32));
}
PG_HD double car_u32_to_uniform(uint32_t w) { return (double)w * (1.0 / 4294967296.0); }
// Feistel network over [0, 2^m), m = bits of n - 1 (at least 2), halves of a = m / 2 and m - a bits: even rounds
// XOR the low half with F(high half), odd rounds the high half with F(low half); cycle-walked into [0, n).
PG_HD int feistel_bits(int n) { int m = 2; while ((1 << m) < n) m++; return m; }
PG_HD uint32_t feistel_mix(uint32_t x, uint32_t k) {
  uint32_t t = (x ^ k) * 0x9E3779B1u;
  t ^= t >> 15; t *= 0x85EBCA6Bu; t ^= t >> 13;
  return t;
}
// position of initial car `slot` among n lane squares (n >= 1, slot < n)
PG_HD int initial_car_position(const uint32_t keys[4], int m, int n, int slot) {
  const int a = m >> 1, b = m - a;
  const uint32_t ma = (1u << a) - 1u, mb = (1u << b) - 1u;
  uint32_t v = (uint32_t)slot;
  do {
    uint32_t lo = v & ma, hi = v >> a;
    lo ^= feistel_mix(hi, keys[0]) & ma;
    hi ^= feistel_mix(lo, keys[1]) & mb;
    lo ^= feistel_mix(hi, keys[2]) & ma;
    hi ^= feistel_mix(lo, keys[3]) & mb;
    v = hi << a | lo;
  } while (v >= (uint32_t)n);
  return (int)v;
}

// Philox word stream (specification shared with the oracle): for a given (stream, tick, episode)
// the 32-bit words come from consecutive Philox4x32-10 blocks, block b = philox(counter =
// (b, tick, episode, stream), key = env seed), 4 words per block. An index draw takes ONE word
// ((word * n) >> 32); a double takes TWO consecutive words ((w0 >> 5) * 2^26 + (w1 >> 6)) / 2^53.
template <int RNG>
struct Rng {
  const DevPtrs& p;
  EnvRegs& e;
  int env;
  uint32_t kcount[5];  // words consumed per stream this tick
  uint32_t b0, b1, b2, b3, cur_block;
  int cur_stream;
  PcgState pcg;        // numpy mode: the stream currently held in registers
  bool pcg_dirty;
  PG_MEMBER Rng(const DevPtrs& p_, EnvRegs& e_, int env_) : p(p_), e(e_), env(env_) {
#pragma unroll
    for (int i = 0; i < 5; i++) kcount[i] = 0;
    cur_stream = -1; cur_block = 0; b0 = b1 = b2 = b3 = 0;
    pcg_dirty = false;
  }
  // ---- numpy mode: stream residency --------------------------------------------------------------
  // The map stream of an episode is a pure function of (seed, episode) and lives only while the map
  // is built; the car / ice / broken-road / sand streams persist in HBM (p.pcg) across ticks.
  PG_MEMBER void np_release() {
    if (cur_stream > 0 && pcg_dirty) p.pcg[(size_t)(cur_stream - 1) * p.pcg_stride + env] = pcg;
    pcg_dirty = false;
  }
  PG_MEMBER void np_acquire(int stream) {
    if (cur_stream == stream) return;
    np_release();
    if (stream == PGTG_STREAM_MAP) pcg_seed_child(p.key[env], 5u * (e.episode - 1u), pcg);
    else pcg = p.pcg[(size_t)(stream - 1) * p.pcg_stride + env];
    cur_stream = stream;
  }
  // seed the four persistent streams of the episode that starts now (children 5r+1 .. 5r+4)
  PG_MEMBER void np_begin_episode() {
    np_release();
    cur_stream = -1;
    uint64_t seed = p.key[env];
    for (int s = 1; s < 5; s++) {
      PcgState st;
      pcg_seed_child(seed, 5u * (e.episode - 1u) + (uint32_t)s, st);
      p.pcg[(size_t)(s - 1) * p.pcg_stride + env] = st;
    }
  }
  // must be called before the Rng goes out of scope (no-op outside numpy mode)
  PG_MEMBER void flush() { if (RNG == PGTG_RNG_NUMPY) { np_release(); cur_stream = -1; } }

  PG_MEMBER uint32_t word(int stream) {
    uint32_t pos = kcount[stream]++;
    uint32_t b = pos >> 2;
    if (stream != cur_stream || b != cur_block) {
      uint64_t key = p.key[env];  // loaded on refill only: most ticks draw nothing
      b0 = b; b1 = e.elapsed; b2 = e.episode; b3 = (uint32_t)stream;
      philox4x32_10(b0, b1, b2, b3, (uint32_t)key, (uint32_t)(key >> 32));
      cur_stream = stream; cur_block = b;
    }
    uint32_t j = pos & 3u;
    return j == 0 ? b0 : j == 1 ? b1 : j == 2 ? b2 : b3;
  }
  // block `b` of a stream (words 4b .. 4b+3), for callers that walk a stream a block at a time and account for the
  // words themselves (set_position afterwards)
  PG_MEMBER void block(int stream, uint32_t b, uint32_t (&w)[4]) {
    const uint64_t key = p.key[env];
    w[0] = b; w[1] = e.elapsed; w[2] = e.episode; w[3] = (uint32_t)stream;
    philox4x32_10(w[0], w[1], w[2], w[3], (uint32_t)key, (uint32_t)(key >> 32));
  }
  PG_MEMBER uint32_t position(int stream) const { return kcount[stream]; }
  PG_MEMBER void set_position(int stream, uint32_t pos) { kcount[stream] = pos; if (cur_stream == stream) cur_stream = -1; }
  // ---- car stream (see the CW_* specification above); tape / numpy modes keep the reference's sequential order
  PG_MEMBER uint32_t car_word(int slot, int pos) {
    const int tag = 0x100 + slot;
    const uint32_t b = (uint32_t)pos >> 2;
    if (cur_stream != tag || cur_block != b) {
      uint32_t w[4];
      philox_car_block(p.key[env], e.elapsed, e.episode, slot, b, w);
      b0 = w[0]; b1 = w[1]; b2 = w[2]; b3 = w[3];
      cur_stream = tag; cur_block = b;
    }
    const int j = pos & 3;
    return j == 0 ? b0 : j == 1 ? b1 : j == 2 ? b2 : b3;
  }
  PG_MEMBER double car_uniform(int slot, int pos) {
    if (RNG != PGTG_RNG_PHILOX) return uniform(PGTG_STREAM_CAR);
    return car_u32_to_uniform(car_word(slot, pos));
  }
  PG_MEMBER int car_index(int slot, int pos, int n) {
    if (n <= 1) return 0;
    if (RNG != PGTG_RNG_PHILOX) return index(PGTG_STREAM_CAR, n);
    return (int)pg_umulhi(car_word(slot, pos), (uint32_t)n);
  }
  PG_MEMBER int car_choice_cdf(int slot, int pos, const double* cdf, int n) {
    if (RNG != PGTG_RNG_PHILOX) return choice_cdf(PGTG_STREAM_CAR, cdf, n);
    double u = car_uniform(slot, pos);
    int i = 0;
    while (i < n - 1 && cdf[i] <= u) i++;
    return i;
  }
  PG_MEMBER double tape_next(int stream, int kind) {
    if (e.cursor >= p.tape_end[env]) { e.err |= 1; return 0.0; }
    if (p.tape_tags[e.cursor] != (uint8_t)(stream * 8 + kind)) e.err |= 2;
    return p.tape_values[e.cursor++];
  }
  // Generator.random()
  PG_MEMBER double uniform(int stream) {
    if (RNG == PGTG_RNG_TAPE) return tape_next(stream, PGTG_DRAW_DOUBLE);
    if (RNG == PGTG_RNG_NUMPY) {
      np_acquire(stream); pcg_dirty = true;
      return pg_dmul((double)(pcg_next64(pcg) >> 11), 1.0 / 9007199254740992.0);
    }
    uint32_t w0 = word(stream), w1 = word(stream);
    // (a * 2^26 + b) / 2^53: every step is exact in float64, so scaling by 2^-53 equals the division
    return pg_dmul(pg_dadd(pg_dmul((double)(w0 >> 5), 67108864.0), (double)(w1 >> 6)), 1.0 / 9007199254740992.0);
  }
  // Generator.integers(0, n) / choice over n items; nothing is consumed for n == 1
  PG_MEMBER int index(int stream, int n) {
    if (n <= 1) return 0;
    if (RNG == PGTG_RNG_TAPE) {
      int v = (int)tape_next(stream, PGTG_DRAW_INDEX);
      if (v < 0 || v >= n) { e.err |= 4; v = 0; }
      return v;
    }
    if (RNG == PGTG_RNG_NUMPY) {
      np_acquire(stream); pcg_dirty = true;
      return (int)pcg_bounded(pcg, (uint32_t)n - 1u);
    }
    return (int)pg_umulhi(word(stream), (uint32_t)n);
  }
  // numpy mode only: random_bounded_uint64(0, rng_inclusive) on `stream`
  PG_MEMBER uint32_t np_bounded(int stream, uint32_t rng_inclusive) {
    np_acquire(stream); pcg_dirty = true;
    return pcg_bounded(pcg, rng_inclusive);
  }
  // Generator.choice(items, p=...): cdf.searchsorted(u, side="right")
  PG_MEMBER int choice_cdf(int stream, const double* cdf, int n) {
    if (RNG == PGTG_RNG_TAPE) {
      int v = (int)tape_next(stream, PGTG_DRAW_INDEX);
      if (v < 0 || v >= n) { e.err |= 4; v = 0; }
      return v;
    }
    double u = uniform(stream);
    int i = 0;
    while (i < n - 1 && cdf[i] <= u) i++;
    return i;
  }
};

// Level sets (specification shared with the oracle, include/pgtg_b200.h): episode k of env i takes its level and its start
// square from ONE block philox(counter = (0, 0, k, PGTG_STREAM_LEVEL), key_i). Word 0 picks the level, (w0 * M) >> 32 (the
// index draw of every stream); env_index sampling takes (env_id_base + i) mod M instead and leaves word 0 unused. Word 1 picks
// the start square, (w1 * 3) >> 32, drawn only when the start line is labelled "start" (build_map's rule). The counter's
// word 3 = 5 differs from streams 0..4 and, in its low byte, from every car-stream counter STREAM_CAR | (slot + 1) << 8, so
// the block is no other draw's.
PG_HD uint32_t level_draw(const DevCfg& c, uint64_t key, uint32_t episode, int env, uint32_t* start_word) {
  uint32_t w0 = 0u, w1 = 0u, w2 = episode, w3 = (uint32_t)PGTG_STREAM_LEVEL;
  philox4x32_10(w0, w1, w2, w3, (uint32_t)key, (uint32_t)(key >> 32));
  *start_word = w1;
  if (c.level_sampling) {
    const int64_t r = (c.env_id_base + env) % (int64_t)c.num_levels;
    return (uint32_t)(r < 0 ? r + c.num_levels : r);
  }
  return pg_umulhi(w0, (uint32_t)c.num_levels);
}
// MapView::line_labels restricted to the start line: the start tile's exit sd is labelled "start" unless the subgoal label
// (the path leaving through that same exit) came first
PG_HD bool start_line_labelled(unsigned start_td, unsigned plan) {
  const int sd = plan_sd(plan), sg = td_sg(start_td);
  const bool on_goal = plan_sy(plan) == plan_gy(plan) && plan_sx(plan) == plan_gx(plan);
  if (!((td_exits(start_td) >> sd) & 1)) return false;
  return !(sg && !on_goal && sg - 1 == sd);
}

// ---------------------------------------------------------------------------------------------
// Map queries on the packed representation.
struct MapView {
  const DevCfg& c;
  const Lut& L;
  uint16_t* tiles;  // shared memory, this env's T descriptors
  uint32_t plan;
  const uint16_t* edge_tab;      // shared-memory copies of the map-generation tables
  const uint16_t* edge_rev;
  const uint16_t* border_slots;
  uint32_t graph;      // connectivity-table index of the generated map's edge set (valid when graph_valid)
  bool graph_valid;
  uint32_t ng_key = 0xFFFFFFFFu;  // nearest_goal's answer computed beforehand (when ng_pre)
  bool ng_pre = false;
  PG_MEMBER bool inside(int x, int y) const { return !(x < 0 || y < 0 || x >= c.WS || y >= c.HS); }  // map.py:44-47
  PG_MEMBER int start_tile() const { return plan_sy(plan) * c.W + plan_sx(plan); }
  PG_MEMBER int goal_tile() const { return plan_gy(plan) * c.W + plan_gx(plan); }

  // Which exit lines of tile t carry a goal-ish label (parser.py:55-77, applied in that order):
  // returns per-direction label codes packed 4 bits each: 0 none, 1 subgoal, 2 used, 3 start, 4 final
  PG_MEMBER unsigned line_labels(int t, unsigned td) const {
    unsigned lab = 0;
    int ex = td_exits(td), sg = td_sg(td), gt = goal_tile();
    if (sg && t != gt && ((ex >> (sg - 1)) & 1)) lab |= ((td & TD_USED) ? 2u : 1u) << (4 * (sg - 1));
    if (t == start_tile()) { int d = plan_sd(plan); if (((ex >> d) & 1) && !((lab >> (4 * d)) & 15)) lab |= 3u << (4 * d); }
    if (t == gt) { int d = plan_gd(plan); if (((ex >> d) & 1) && !((lab >> (4 * d)) & 15)) lab |= 4u << (4 * d); }
    return lab;
  }
  // features of one square inside the map (the reference's set[str], parser.py:44-155)
  PG_MEMBER unsigned features(int x, int y) const {
    int tx = x / TILE, ty = y / TILE, sq = (x - tx * TILE) * TILE + (y - ty * TILE), t = ty * c.W + tx;
    unsigned td = tiles[t];
    int ex = td_exits(td);
    if (bit81(L.wall[ex], sq)) return SF_WALL;
    unsigned f = 0;
    int ot = td_otype(td);
    if (ot && bit81(L.mask[td_omask(td)], sq)) f |= (SF_ICE >> 1) << ot;  // 1 ice .. 4 light
    if (bit81(L.exit_any, sq) && (td_sg(td) || t == start_tile())) {
      // the square lies on exactly one exit line d: label that line only, in the order of
      // parser.py:55-77 (subgoal, then start, then final goal)
      int d = bit81(L.exit_line[0], sq) ? 0 : bit81(L.exit_line[1], sq) ? 1 : bit81(L.exit_line[2], sq) ? 2 : 3;
      if ((ex >> d) & 1) {
        int sg = td_sg(td), gt = goal_tile();
        if (sg && t != gt && d == sg - 1) f |= (td & TD_USED) ? SF_USED : SF_SUBGOAL;
        else if (t == start_tile() && d == plan_sd(plan)) f |= SF_START;
        else if (t == gt && d == plan_gd(plan)) f |= SF_FINAL;
      }
    }
    return f;
  }
  PG_MEMBER int tile_type_at(int x, int y) const { return td_exits(tiles[(y / TILE) * c.W + x / TILE]); }
  PG_MEMBER int local_sq(int x, int y) const { return (x % TILE) * TILE + (y % TILE); }
  PG_MEMBER bool light_at(int x, int y) const {
    int tx = x / TILE, ty = y / TILE, sq = (x - tx * TILE) * TILE + (y - ty * TILE);
    unsigned td = tiles[ty * c.W + tx];
    return td_otype(td) == 4 && bit81(L.mask[td_omask(td)], sq) && !bit81(L.wall[td_exits(td)], sq);
  }
  // set_subgoals_to_used (map.py:143-171): the flood covers exactly the tile's 3-square exit line
  PG_MEMBER void consume_subgoal(int x, int y) { tiles[(y / TILE) * c.W + x / TILE] |= TD_USED; }

  // nearest remaining subgoal / final-goal square: first strict minimum of the Manhattan distance
  // in the x-major scan (environment.py:1047-1053, 1474-1480) == lexicographic min of (d, x, y), i.e. the minimum of the
  // key d << 16 | x << 8 | y. tile_goal_key = the best key among the goal-line squares of tile t (0xFFFFFFFF: none).
  PG_MEMBER uint32_t tile_goal_key(int t, int px, int py) const { return tile_goal_key(t, (t % c.W) * TILE, (t / c.W) * TILE, px, py); }
  PG_MEMBER uint32_t tile_goal_key(int t, int ox, int oy, int px, int py) const {  // (ox, oy): the tile's origin square
    const unsigned td = tiles[t];
    const int sg = td_sg(td);
    if (!sg) return 0xFFFFFFFFu;
    int d;
    if (t == goal_tile()) { d = plan_gd(plan); if (!((td_exits(td) >> d) & 1)) return 0xFFFFFFFFu; }
    else { if (td & TD_USED) return 0xFFFFFFFFu; d = sg - 1; }
    // claimed earlier by start? (only possible on degenerate fixed maps) -- labels decide
    const unsigned lab = (line_labels(t, td) >> (4 * d)) & 15;
    if (lab != 1 && lab != 4) return 0xFFFFFFFFu;
    uint32_t best = 0xFFFFFFFFu;
#pragma unroll
    for (int k = 0; k < 3; k++) {  // the 3 squares of exit line d (north (3..5,0) east (8,3..5) ...), from the derived LUT
      const int xy = L.line_xy[d][k];
      const int X = ox + (xy & 15), Y = oy + (xy >> 4);
      const uint32_t key = (uint32_t)(abs(X - px) + abs(Y - py)) << 16 | (uint32_t)X << 8 | (uint32_t)Y;
      best = key < best ? key : best;
    }
    return best;
  }
  PG_MEMBER bool nearest_goal(int px, int py, int& gx, int& gy) const {
    uint32_t best = ng_key;  // (the traffic tick computes the key beforehand, one tile per thread)
    if (!ng_pre) {
      best = 0xFFFFFFFFu;
      int ox = 0, oy = 0;  // tile origins walked row by row (no division per tile)
      for (int t = 0; t < c.T; t++) {
        const uint32_t k = tile_goal_key(t, ox, oy, px, py);
        best = k < best ? k : best;
        ox += TILE;
        if (ox == c.WS) { ox = 0; oy += TILE; }
      }
    }
    gx = (int)((best >> 8) & 255u); gy = (int)(best & 255u);
    return best != 0xFFFFFFFFu;
  }
};

}  // namespace pgtg
