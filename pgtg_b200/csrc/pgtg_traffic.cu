// pgtg_traffic.cu -- the traffic tick kernel (phases in pgtg_traffic.cuh) and its launch code.
//
// One CTA = G consecutive envs (G = 32) and NT threads; the CTA alternates between "flat over the cars of
// its envs" and "one env per thread" with a barrier in between (see the header). Outputs and state layout
// are those of the sequential tick, so reset / observe / state dumps keep using the general kernel.
#include <cuda_runtime.h>
#include <stdlib.h>

#include "pgtg_env.hpp"
#include "pgtg_traffic.cuh"

namespace pgtg {

struct TkStats { double* rows; };

template <int TMAX, bool PREGEN, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) pgtg_traffic_tick_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p,
                                                                      const void* __restrict__ actions, int action_bytes, TkStats sa,
                                                                      const __grid_constant__ TkLayout layout) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int G = layout.G;
  const int env0 = blockIdx.x * G;
  const int nvalid = min(G, c.N - env0);
  const TkShared sh = tk_carve(smem, layout);
  BlockShared bs;  // the parts the shared phases (stage, expand) use
  bs.lut = sh.lut; bs.spread = sh.spread; bs.tiles = sh.tiles; bs.bits = sh.bits; bs.bits_words = sh.bits_words; bs.done_list = sh.done_list;
  bs.regs = nullptr; bs.counters = sh.counters; bs.dsum = sh.dsum; bs.edge_tab = bs.edge_rev = bs.border_slots = nullptr;

  // ---- stage ---------------------------------------------------------------------------------------
  phase_stage(c, p, bs, tid, NT, env0, nvalid, true, false);
  for (int i = tid; i < G * sh.occ_words; i += NT) sh.occ[i] = 0;
  if (tid < 16) sh.counters[tid] = 0;
  for (int i = tid; i < 32 * 32; i += NT) sh.wbits[i] = 0;
  for (int i = tid; i < c.T; i += NT) tk_stage_tile(c, sh, i);
  if (tid < 2) sh.dsum[tid] = 0.0;
  const bool mine = tid < nvalid;
  const int env = env0 + tid;
  if (mine) {
    const int a = action_bytes == 8 ? (int)((const long long*)actions)[env] : ((const int*)actions)[env];
    tk_stage_env(c, p, sh, tid, env, a);
  }
  __syncthreads();
  if (mine) tk_prefix(sh, sh.off, tid, nvalid, false);
  if (c.num_rules > 0)  // the rule engine's heading needs the nearest goal-line square of the position before the move
    for (int i = tid; i < nvalid * c.T; i += NT) tk_goal_key(c, sh, i / c.T, i % c.T, false);
  __syncthreads();
  const int total = sh.off[G];

  // ---- the cars: intents (flat), then blocking in list order + commit (one env per warp) ---------------------
  for (int item = tid; item < total; item += NT) {
    const int g = sh.item_g[item];
    tk_intent(c, p, sh, g, item - sh.off[g], env0 + g);
  }
  __syncthreads();
  for (int g = tid >> 5; g < nvalid; g += NT >> 5)  // one env per warp, 32 cars per step
    if (sh.env[g].n_cars > 0) tk_resolve_commit(c, p, sh, g, env0 + g, tid >> 5);
  __syncthreads();

  // ---- the agent --------------------------------------------------------------------------------------
  StepResult r;
  r.outcome = 0; r.ep_return = 0; r.ep_disc = 0;
  int len = 0;
  if (mine) { r = tk_agent(c, p, sh, tid, env); len = r.outcome ? (int)sh.env[tid].e.elapsed : 0; sh.env[tid].ng_key = 0xFFFFFFFFu; }
  const bool done = r.outcome != 0;
  if (tid < ((G + 31) & ~31)) {  // warps that hold envs: episode statistics and the map requests of the finished ones
    const unsigned any = __ballot_sync(0xffffffffu, done);
    if (any) {
      const unsigned g2 = __ballot_sync(0xffffffffu, r.outcome == 2), cr = __ballot_sync(0xffffffffu, r.outcome == 1),
                     tr = __ballot_sync(0xffffffffu, r.outcome == 3);
      const int lsum = __reduce_add_sync(0xffffffffu, len);
      double rs = r.ep_return;
      for (int o = 16; o > 0; o >>= 1) rs += __shfl_down_sync(0xffffffffu, rs, o);
      uint32_t qbase = 0;
      int lbase = 0;
      if (lane == 0) {
        atomicAdd(&sh.counters[8], __popc(g2)); atomicAdd(&sh.counters[9], __popc(cr)); atomicAdd(&sh.counters[10], __popc(tr));
        atomicAdd(&sh.counters[11], lsum);
        lbase = atomicAdd(&sh.counters[12], __popc(any));
        atomicAdd(&sh.dsum[0], rs);
        if (PREGEN) qbase = atomicAdd(p.regen_count + p.parity, (uint32_t)__popc(any));
      }
      if (c.eval_on) {
        const unsigned neg = __ballot_sync(0xffffffffu, done && r.ep_disc < 0);
        double ds = r.ep_disc;
        for (int o = 16; o > 0; o >>= 1) ds += __shfl_down_sync(0xffffffffu, ds, o);
        if (lane == 0) { atomicAdd(&sh.dsum[1], ds); atomicAdd(&sh.counters[13], __popc(neg)); }
      }
      qbase = __shfl_sync(0xffffffffu, qbase, 0);
      lbase = __shfl_sync(0xffffffffu, lbase, 0);
      if (done) {
        const int k = __popc(any & ((1u << lane) - 1u));
        sh.done_list[lbase + k] = tid;
        if (PREGEN) {  // the episode about to start frees ring slot (k & 1): ask for the map of episode k + 2
          uint2 q; q.x = (uint32_t)env; q.y = sh.env[tid].e.episode + 3u;
          p.regen_list[(size_t)p.parity * 2 * c.N + qbase + k] = q;
        }
      }
    }
  }
  __syncthreads();
  const int n_done = sh.counters[12];

  // ---- terminal observation of the finished envs (optional output) ------------------------------------------
  if (c.write_final_obs && n_done) {  // CTA-uniform
    if (c.use_nsd) {  // next_subgoal_direction of the terminal observation
      for (int i = tid; i < nvalid * c.T; i += NT) if (sh.env[i / c.T].done) tk_goal_key(c, sh, i / c.T, i % c.T, true);
      __syncthreads();
    }
    for (int item = tid; item < total; item += NT) {
      const int g = sh.item_g[item];
      const TEnv& t = sh.env[g];
      if (t.done) tk_car_bit(c, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, t.e.x, t.e.y, sh.fxy[g * sh.MC + item - sh.off[g]]);
    }
    if (c.sliding)
      for (int i = tid; i < nvalid * c.C * c.P; i += NT) if (sh.env[i / (c.C * c.P)].done) tk_sliding_column(c, sh, i / (c.C * c.P), i % (c.C * c.P));
    if (done) { tk_emit(c, p, sh, tid, env, true); sh.env[tid].ng_key = 0xFFFFFFFFu; }
    __syncthreads();
    phase_expand_final(c, p.f_obs_map, bs, tid, NT, env0, n_done);
    __syncthreads();
    for (int i = tid; i < sh.bits_words; i += NT) sh.bits[i] = 0;
    __syncthreads();
  }

  // ---- traffic plane of the running envs (flat) ------------------------------------------------------------------
  for (int item = tid; item < total; item += NT) {
    const int g = sh.item_g[item];
    const TEnv& t = sh.env[g];
    if (!t.done) tk_car_bit(c, sh.bits, (uint32_t)g * (uint32_t)c.obs_bits, t.e.x, t.e.y, sh.fxy[g * sh.MC + item - sh.off[g]]);
  }

  // ---- same-step auto-reset: the map (per env), then the new episode's cars (flat) ------------------------------
  if (n_done) {
    if (done) tk_reset_map<TMAX, PREGEN>(c, p, sh, tid, env);
    __syncthreads();
    if (NT >= 3 * G) {  // lane squares, spawner list and placement keys of the new maps: three groups of warps side by side
      const int part = tid / G, g = tid - part * G;
      if (part < 3 && g < nvalid && sh.env[g].done) tk_reset_traffic(c, p, sh, g, env0 + g, 1 << part);
    } else if (done) tk_reset_traffic(c, p, sh, tid, env, 7);
    __syncthreads();
    if (mine) tk_prefix(sh, sh.off2, tid, nvalid, true);  // (rewrites the item table: the tick's items are done with)
    __syncthreads();
    const int total2 = sh.off2[G];
    for (int item = tid; item < total2; item += NT) {
      const int g = sh.item_g[item];
      tk_new_car(c, p, sh, g, item - sh.off2[g], env0 + g);
    }
  }

  // ---- map planes + scalars + state (per env) ---------------------------------------------------------------------
  if (c.use_nsd) {  // next_subgoal_direction: nearest goal-line square of the observed position, one tile per thread
    for (int i = tid; i < nvalid * c.T; i += NT) tk_goal_key(c, sh, i / c.T, i % c.T, true);
    __syncthreads();
  }
  if (c.sliding)  // sliding-window planes, one (plane, column) per thread
    for (int i = tid; i < nvalid * c.C * c.P; i += NT) tk_sliding_column(c, sh, i / (c.C * c.P), i % (c.C * c.P));
  if (mine) tk_emit(c, p, sh, tid, env, false);
  __syncthreads();
  if (tid == 0 && n_done) {
    double* row = sa.rows + (size_t)blockIdx.x * STATS_STRIDE;
    row[0] += n_done; row[1] += sh.dsum[0]; row[2] += sh.counters[11];
    row[3] += sh.counters[8]; row[4] += sh.counters[9]; row[5] += sh.counters[10];
    if (c.eval_on) { row[6] += sh.dsum[1]; row[7] += sh.counters[13]; }
  }
  phase_expand(c, p.obs_map, bs, tid, NT, env0, nvalid, p.obs_packed);
}

}  // namespace pgtg

// Geometry of the traffic tick for a configuration: envs per CTA (a multiple of 32: every CTA's slice of the
// observation planes must start 32-byte aligned), threads per CTA and dynamic shared memory; G = 0 when the
// per-env working set does not fit (very large maps with dense traffic): the sequential tick runs instead.
int pgtg_traffic_geometry(const pgtg::DevCfg& c, int* G, int* NT, size_t* smem) {
  int g = 32;
  const char* forced_g = getenv("PGTG_TRAFFIC_G");  // experiment knob: 32 / 64 / 128 envs per CTA
  if (forced_g && (atoi(forced_g) == 32 || atoi(forced_g) == 64 || atoi(forced_g) == 128)) g = atoi(forced_g);
  const pgtg::TkLayout L = pgtg::tk_layout(c, g);
  *G = 0; *NT = 0; *smem = 0;
  if (!pgtg::tk_fits(c, g)) return 0;
  *G = g; *smem = L.total;
  // the per-env phases keep one warp per CTA busy: small CTAs (many per SM) while shared memory allows, one big CTA otherwise
  *NT = L.total > 72u * 1024u ? 1024 : (L.total > 28u * 1024u ? 256 : 128);
  const char* forced = getenv("PGTG_TRAFFIC_NT");  // experiment knob
  if (forced && (atoi(forced) == 64 || atoi(forced) == 128 || atoi(forced) == 256 || atoi(forced) == 1024)) *NT = atoi(forced);
  if (*NT < g) *NT = g;  // one env per thread in the per-env phases
  return 1;
}

template <int TMAX, bool PREGEN, int NT, int MINB>
static int launch_traffic(pgtg_env* e, const void* actions, int action_bytes, cudaStream_t st) {
  auto kern = pgtg::pgtg_traffic_tick_kernel<TMAX, PREGEN, NT, MINB>;
  const pgtg::TkLayout L = pgtg::tk_layout(e->dc, e->traffic_G);
  static bool attr_set = false;
  if (!attr_set) {
    // same carveout as the map-generation kernel so that the two can share an SM (pgtg_tick_kernels.cuh)
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    attr_set = true;
  }
  if (L.total > 48u * 1024u) {
    cudaError_t rc = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
    if (rc != cudaSuccess) return (int)rc;
  }
  pgtg::TkStats sa = {e->stats_rows};
  const int grid = (e->dc.N + L.G - 1) / L.G;
  kern<<<grid, NT, L.total, st>>>(e->dc, e->dp, actions, action_bytes, sa, L);
  return (int)cudaGetLastError();
}

template <int TMAX, bool PREGEN>
static int launch_traffic_nt(pgtg_env* e, const void* actions, int action_bytes, cudaStream_t st) {
  if (e->traffic_NT == 1024) return launch_traffic<TMAX, PREGEN, 1024, 1>(e, actions, action_bytes, st);
  if (e->traffic_NT == 128) return launch_traffic<TMAX, PREGEN, 128, 8>(e, actions, action_bytes, st);
  if (e->traffic_NT == 64) return launch_traffic<TMAX, PREGEN, 64, 16>(e, actions, action_bytes, st);
  return launch_traffic<TMAX, PREGEN, 256, 3>(e, actions, action_bytes, st);
}

int pgtg_launch_traffic_tick(pgtg_env* e, const void* actions, int action_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (e->dc.pregen) return launch_traffic_nt<16, true>(e, actions, action_bytes, st);
  if (e->dc.T <= 16) return launch_traffic_nt<16, false>(e, actions, action_bytes, st);
  if (e->dc.T <= 64) return launch_traffic_nt<64, false>(e, actions, action_bytes, st);
  return launch_traffic_nt<256, false>(e, actions, action_bytes, st);
}
