// pgtg_tick_kernels.cuh -- the fused tick kernel, the map-generation kernel and their launch code, as
// templates over the random-number source. Instantiated once per RNG mode in pgtg_inst_*.cu so that the
// three families compile in parallel; pgtg_kernels.cu dispatches to them.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "pgtg_env.hpp"

namespace pgtg {

#ifndef PGTG_MIN_BLOCKS
#define PGTG_MIN_BLOCKS 8
#endif
#ifndef PGTG_MAPGEN_TABLED_MIN_BLOCKS
#define PGTG_MAPGEN_TABLED_MIN_BLOCKS 12  /* 40 registers (the staged tabled generator: numpy-exact mode, 9-tile maps); at 16 CTAs/SM it spills */
#endif
#ifndef PGTG_LEAN_MIN_BLOCKS
#define PGTG_LEAN_MIN_BLOCKS 8
#endif
// bytes of the per-thread edge array of the register-resident map generation: 7 words, an odd stride, so that the lanes of
// a warp reading the same index hit 32 different banks
#define PGTG_EDGE_ROW 28
#ifndef PGTG_MAPGEN_MIN_BLOCKS
#define PGTG_MAPGEN_MIN_BLOCKS 12
#endif

// per-CTA episode statistics row (no cross-CTA atomics on the hot path)
struct StatsArgs {
  double* rows;  // [gridDim.x][8]
};

// -DPGTG_PHASE_CLOCKS: profiling build (never the shipped one; load it through PGTG_B200_LIB):
// per-warp SM-clock time of each phase of the ring-fed tick, summed into g_phase_clk and printed
// by the statistics reduction. The macros expand to nothing in the normal build.
#ifdef PGTG_PHASE_CLOCKS
__device__ unsigned long long g_phase_clk[16];
#define PG_CLK_INIT long long clk_prev = clock64();
#define PG_CLK(i) { if ((threadIdx.x & 31) == 0) { long long t_ = clock64(); atomicAdd(&g_phase_clk[i], (unsigned long long)(t_ - clk_prev)); clk_prev = t_; } }
#else
#define PG_CLK_INIT
#define PG_CLK(i)
#endif

// (FINAL: the lean instantiation that also writes the terminal observation of the finished envs, gymnasium's final_observation;
//  SLIDE: the lean instantiation for the sliding window and / or next_subgoal_direction -- the observation of train.py without cars)
//  INLINE: a finished env's thread rebuilds the ring slot it has just consumed right here, after the expansion, instead of queueing
//  a request for the map-generation kernel (register-resident generator; experiment, DESIGN.md 7)
template <int RNG, int MODE, int TMAX, bool PREGEN, bool LEAN = false, bool FINAL = false, bool SLIDE = false, bool INLINE = false>
__global__ void __launch_bounds__(128, LEAN ? PGTG_LEAN_MIN_BLOCKS : PGTG_MIN_BLOCKS) pgtg_tick_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p,
                                                        const uint8_t* __restrict__ mask, const int64_t* __restrict__ seeds,
                                                        const void* __restrict__ actions, int action_bytes, StatsArgs sa,
                                                        const __grid_constant__ SharedLayout layout) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int B = blockDim.x, tid = threadIdx.x;
  const int env0 = blockIdx.x * B;
  const int nvalid = min(B, c.N - env0);
  const int env = env0 + tid;
  const bool valid = tid < nvalid;
  const int lane = tid & 31, warp = tid >> 5, nwarps = B >> 5;
  BlockShared sh = carve_layout(smem, layout);

  PG_CLK_INIT
  phase_stage(c, p, sh, tid, B, env0, nvalid, true, !(PREGEN && MODE == MODE_STEP));
  if (tid < 8) { sh.counters[8 + tid] = 0; sh.dsum[tid] = 0.0; }
  PG_CLK(0)
  __syncthreads();
  PG_CLK(1)

  bool done = false;
  if (MODE == MODE_STEP) {
    StepResult r;
    r.outcome = 0; r.ep_return = 0; r.ep_disc = 0;
    int len = 0;
    EnvRegs er;  // lean instantiation: the env's registers stay in registers from step to emit
    if (valid) {
      int a = action_bytes == 8 ? (int)((const long long*)actions)[env] : ((const int*)actions)[env];
      if (LEAN) { r = phase_step_regs<RNG, true>(c, p, sh, tid, env, a, er); len = (int)er.elapsed; }
      else { r = phase_step<RNG, false>(c, p, sh, tid, env, a); len = (int)sh.regs[tid].elapsed; }
      done = r.outcome != 0;
      len = done ? len : 0;
    }
    PG_CLK(2)
    // episode statistics: ballots for the counters, warp reductions for the sums, one row per CTA
    unsigned any = __ballot_sync(0xffffffffu, done);
    if (any) {
      unsigned g = __ballot_sync(0xffffffffu, r.outcome == 2), cr = __ballot_sync(0xffffffffu, r.outcome == 1),
               tr = __ballot_sync(0xffffffffu, r.outcome == 3);
      int lsum = __reduce_add_sync(0xffffffffu, len);
      double rs = r.ep_return;
      for (int o = 16; o > 0; o >>= 1) rs += __shfl_down_sync(0xffffffffu, rs, o);
      if (lane == 0) {
        atomicAdd(&sh.counters[8], __popc(g)); atomicAdd(&sh.counters[9], __popc(cr)); atomicAdd(&sh.counters[10], __popc(tr));
        atomicAdd(&sh.counters[11], lsum); atomicAdd(&sh.counters[12], __popc(any));
        atomicAdd(&sh.dsum[0], rs);
      }
      if (c.eval_on) {  // evaluator statistics: sum of discounted returns, episodes with a negative one
        const unsigned neg = __ballot_sync(0xffffffffu, done && r.ep_disc < 0);
        double ds = r.ep_disc;
        for (int o = 16; o > 0; o >>= 1) ds += __shfl_down_sync(0xffffffffu, ds, o);
        if (lane == 0) { atomicAdd(&sh.dsum[1], ds); atomicAdd(&sh.counters[13], __popc(neg)); }
      }
    }
    if (LEAN || (PREGEN && !c.write_final_obs)) {  // (LEAN && FINAL is the one lean case with terminal observations)
      // Hot configuration (next maps come from the ring, no terminal-observation output): the
      // reset is a cheap swap, so every finished env is reset by its own thread and the CTA
      // needs one barrier only, the one in front of the byte expansion. Map requests are queued
      // per warp; the atomic's round trip hides behind the observation emit.
      uint32_t k = 0, qbase = 0;
      if (!INLINE && any && lane == 0) qbase = atomicAdd(p.regen_count + p.parity, (uint32_t)__popc(any));
      PG_CLK(3)
      if (LEAN && FINAL) {  // terminal observation first: emit the finished envs' planes, expand their rows, clear the bitstring
        if (lane == 0) sh.counters[16 + warp] = (int)any;
        if (done) phase_emit_regs<true, SLIDE>(c, p, sh, tid, env, true, er);
        __syncthreads();
        phase_expand_final_vec(c, p.f_obs_map, sh, tid, B, env0, nvalid, sh.counters + 16, p.f_obs_packed);
        __syncthreads();
        {
          uint4 z; z.x = z.y = z.z = z.w = 0;
          uint4* b4 = (uint4*)sh.bits;
          for (int i = tid; i < sh.bits_words / 4; i += B) b4[i] = z;
          for (int i = (sh.bits_words / 4) * 4 + tid; i < sh.bits_words; i += B) sh.bits[i] = 0;
        }
        __syncthreads();
      }
      if (done) {
        if (LEAN) { k = er.episode + 1u; phase_reset_regs<RNG, TMAX, true, true>(c, p, sh, tid, env, er); }
        else { k = sh.regs[tid].episode + 1u; phase_reset<RNG, TMAX, true, false>(c, p, sh, tid, env); }  // k: the episode this env is about to start
      }
      PG_CLK(4)
      if (valid) { if (LEAN) phase_emit_regs<true, SLIDE>(c, p, sh, tid, env, false, er); else phase_emit<false>(c, p, sh, tid, env, false); }
      PG_CLK(5)
      if (!INLINE && any) {
        qbase = __shfl_sync(0xffffffffu, qbase, 0);
        if (done) {
          uint2 q; q.x = (uint32_t)env; q.y = k + 2u;
          p.regen_list[(size_t)p.parity * 2 * c.N + qbase + __popc(any & ((1u << lane) - 1u))] = q;
        }
      }
      PG_CLK(6)
      __syncthreads();
      PG_CLK(7)
      if (tid == 0 && sh.counters[12]) {
        double* row = sa.rows + (size_t)blockIdx.x * STATS_STRIDE;
        row[0] += sh.counters[12]; row[1] += sh.dsum[0]; row[2] += sh.counters[11];
        row[3] += sh.counters[8]; row[4] += sh.counters[9]; row[5] += sh.counters[10];
        if (c.eval_on) { row[6] += sh.dsum[1]; row[7] += sh.counters[13]; }
      }
      phase_expand(c, p.obs_map, sh, tid, B, env0, nvalid, p.obs_packed);
      PG_CLK(8)
      if (INLINE && LEAN && done)  // (the thread's tile row is dead after the emit: it serves as the generator's edge array)
        phase_pregenerate_in_registers<RNG>(c, p, (uint8_t*)(sh.tiles + tid * c.tile_stride), env, k + 2u);
      return;
    }
  } else if (MODE == MODE_RESET) {
    if (valid) {
      EnvRegs e = load_regs(c, p, env);
      if (!mask || mask[env]) {
        if (seeds) { p.key[env] = (uint64_t)seeds[env]; e.episode = 0; }
        p.ep_return[env] = 0.0;
        if (p.ep_disc) p.ep_disc[env] = 0.0;
        done = true;
      }
      sh.regs[tid] = e;
    }
  } else {
    if (valid) sh.regs[tid] = load_regs(c, p, env);
  }

  if (LEAN) return;  // (the lean instantiation is step-mode only and has returned above)

  // compaction of the done envs: warp ballot + CTA scan -> dense list in shared memory
  unsigned ballot = __ballot_sync(0xffffffffu, done);
  if (lane == 0) sh.counters[1 + warp] = __popc(ballot);
  __syncthreads();
  int base = 0, n_done = 0;
  for (int w = 0; w < nwarps; w++) { int v = sh.counters[1 + w]; if (w < warp) base += v; n_done += v; }
  if (done) sh.done_list[base + __popc(ballot & ((1u << lane) - 1u))] = tid;
  if (MODE == MODE_STEP && tid == 0 && n_done) {
    double* row = sa.rows + (size_t)blockIdx.x * STATS_STRIDE;
    row[0] += n_done; row[1] += sh.dsum[0]; row[2] += sh.counters[11];
    row[3] += sh.counters[8]; row[4] += sh.counters[9]; row[5] += sh.counters[10];
    if (c.eval_on) { row[6] += sh.dsum[1]; row[7] += sh.counters[13]; }
  }
  __syncthreads();

  if (MODE != MODE_OBSERVE && c.pregen && n_done) {
    // CTA-uniform: queue map requests for the map-generation kernel. An env that starts episode k
    // frees ring slot (k & 1): ask for the map of episode k + 2 (a full reset also needs k + 1).
    const int per = MODE == MODE_RESET ? 2 : 1;
    if (tid == 0) sh.counters[20] = (int)atomicAdd(p.regen_count + p.parity, (uint32_t)(n_done * per));
    __syncthreads();
    if (tid < n_done) {
      int local = sh.done_list[tid];
      uint32_t k = sh.regs[local].episode + 1u;  // the episode this env is about to start
      uint2* q = p.regen_list + (size_t)p.parity * 2 * c.N + sh.counters[20] + tid * per;
      uint2 r; r.x = (uint32_t)(env0 + local);
      if (MODE == MODE_RESET) { r.y = k + 1u; q[0] = r; r.y = k + 2u; q[1] = r; }
      else { r.y = k + 2u; q[0] = r; }
    }
  }

  if (MODE == MODE_STEP && c.write_final_obs && n_done) {  // CTA-uniform condition
    if (done) phase_emit(c, p, sh, tid, env, true);
    __syncthreads();
    phase_expand_final(c, p.f_obs_map, sh, tid, B, env0, n_done, p.f_obs_packed, nvalid);
    __syncthreads();
    for (int i = tid; i < sh.bits_words; i += B) sh.bits[i] = 0;
    __syncthreads();
  }

  if (MODE != MODE_OBSERVE) {
    if (tid < n_done) {
      int local = sh.done_list[tid];
      phase_reset<RNG, TMAX, PREGEN>(c, p, sh, local, env0 + local);
    }
    __syncthreads();
  }
  if (valid) phase_emit(c, p, sh, tid, env, false);
  __syncthreads();
  phase_expand(c, p.obs_map, sh, tid, B, env0, nvalid, p.obs_packed);
}

// Map generation ahead of time: dense over the envs queued by the tick that just ran (every lane
// busy, no CTA barrier after the staging, tiny shared-memory footprint -> high occupancy). The
// loop is grid-stride so that the launch code may also run it as a small persistent grid
// (PGTG_MAPGEN_CTAS_PER_SM); the default is one request per thread. TABLED: see generate_map.
template <int RNG, int TMAX, bool TABLED = false>
__global__ void __launch_bounds__(128, TABLED ? PGTG_MAPGEN_TABLED_MIN_BLOCKS : PGTG_MAPGEN_MIN_BLOCKS) pgtg_mapgen_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, int parity,
                                                                                const __grid_constant__ SharedLayout layout) {
  extern __shared__ __align__(16) unsigned char smem[];
  const uint32_t count = p.regen_count[parity];
  if (blockIdx.x * blockDim.x >= count) return;
  const uint2* list = p.regen_list + (size_t)parity * 2 * c.N;
  BlockShared sh = carve_layout(smem, layout);
  stage_tables(c, p, sh, threadIdx.x, blockDim.x);
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    uint2 r = list[i];
    phase_pregenerate<RNG, TMAX, TABLED>(c, p, sh, threadIdx.x, (int)r.x, r.y);
  }
}

// The same for configurations whose map is assembled in registers (map_in_registers -- the headline configuration): no
// staged tables, no barrier; shared memory holds only each thread's edge array. Its own kernel so that the register
// allocation is not the staged path's (MINB CTAs of 128 threads per SM; measured, see DESIGN.md 7).
template <int RNG, int MINB>
__global__ void __launch_bounds__(128, MINB) pgtg_mapgen_registers_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, int parity) {
  extern __shared__ __align__(16) unsigned char smem[];
  const uint32_t count = p.regen_count[parity];
  if (blockIdx.x * blockDim.x >= count) return;
  const uint2* list = p.regen_list + (size_t)parity * 2 * c.N;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint2 r = list[i];
    phase_pregenerate_in_registers<RNG>(c, p, smem + threadIdx.x * PGTG_EDGE_ROW, (int)r.x, r.y);
  }
}

}  // namespace pgtg

// launch code: returns the cudaError_t of the launch (0 = ok)
static inline int lk(cudaError_t e) { return (int)e; }

template <int RNG, int MODE, int TMAX, bool PREGEN, bool LEAN = false, bool FINAL = false, bool SLIDE = false, bool INLINE = false>
static int launch_one(pgtg_env* e, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, cudaStream_t st) {
  auto kern = pgtg::pgtg_tick_kernel<RNG, MODE, TMAX, PREGEN, LEAN, FINAL, SLIDE, INLINE>;
  // same L1/shared carveout as the map-generation kernel: an SM cannot host CTAs of two kernels with
  // different carveouts, which would serialise the two (measured: no overlap at all without this)
  static bool carve_set = false;
  const size_t smem = LEAN ? pgtg::block_shared_bytes(e->dc, e->block, true) : e->smem;
  if (!carve_set) {
    // The lean tick's eight CTAs (19 KB each + 1 KB reserved) fit the 164 KB shared-memory configuration: asking for it instead
    // of the maximum leaves 64 KB more L1 (measured: 0.345 instead of 0.348 ms per tick). Everything else keeps the maximum
    // (lean+slide needs it; the general and traffic ticks share SMs with the staged map generation, same carveout).
    const bool fits164 = LEAN && (smem + 1024) * PGTG_LEAN_MIN_BLOCKS <= 164u * 1024u;
    const char* cv = getenv("PGTG_TICK_CARVEOUT");  // tuning knob (DESIGN.md 7)
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cv ? atoi(cv) : fits164 ? 72 : (int)cudaSharedmemCarveoutMaxShared);
    carve_set = true;
  }
  if (smem > 48 * 1024) {
    { int rc = lk(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); if (rc) return rc; }
  }
  pgtg::StatsArgs sa = {e->stats_rows};
  unsigned char* const origin = (unsigned char*)4096;  // any 16-byte-aligned address: only differences are used
  const pgtg::SharedLayout layout = pgtg::layout_of(pgtg::carve_shared(origin, e->dc, e->block, LEAN), origin);
  kern<<<e->nblk, e->block, smem, st>>>(e->dc, e->dp, mask, seeds, actions, action_bytes, sa, layout);
  return lk(cudaGetLastError());
}

// TMAX = compile-time bound on the tile count (register-resident boards for the default 4x4 map)
template <int RNG, int MODE, bool PREGEN>
static int launch_sized(pgtg_env* e, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, cudaStream_t st) {
  if (e->dc.T <= 16) return launch_one<RNG, MODE, 16, PREGEN>(e, mask, seeds, actions, action_bytes, st);
  if (e->dc.T <= 64) return launch_one<RNG, MODE, 64, PREGEN>(e, mask, seeds, actions, action_bytes, st);
  return launch_one<RNG, MODE, 256, PREGEN>(e, mask, seeds, actions, action_bytes, st);
}

template <int RNG, int MINB>
static int launch_mapgen_registers(pgtg_env* e, cudaStream_t st, int grid, int carveout) {
  auto kern = pgtg::pgtg_mapgen_registers_kernel<RNG, MINB>;
  static bool carve_set = false;
  if (!carve_set) { cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, carveout); carve_set = true; }
  kern<<<grid, 128, 128 * PGTG_EDGE_ROW, st>>>(e->dc, e->dp, e->dp.parity);
  return lk(cudaGetLastError());
}

template <int RNG, int TMAX, bool TABLED = false>
static int launch_mapgen(pgtg_env* e, cudaStream_t st) {
  const int B = 128;
  size_t smem = pgtg::mapgen_shared_bytes(e->dc, B);
  int full = (2 * e->dc.N + B - 1) / B;
  int grid = e->mapgen_grid > 0 && e->mapgen_grid < full ? e->mapgen_grid : full;
  if constexpr (RNG == PGTG_RNG_PHILOX && TABLED) {
    if (pgtg::map_in_registers(e->dc) && !getenv("PGTG_NO_MAP_IN_REGISTERS")) {
      const char* mb = getenv("PGTG_MAPGEN_MINB");   // tuning knobs (DESIGN.md 7)
      const char* cv = getenv("PGTG_MAPGEN_CARVEOUT");
      // 12 CTAs/SM at 40 registers (sweep of 8 / 10 / 12 / 16 on the final kernel: 12 is 1-2 % ahead); 54 KB shared and the rest
      // L1 (the connectivity lookups of the first trips hit it) -- except next to the traffic tick, which leaves SMs free for
      // this kernel only if both ask for the same carveout (measured, DESIGN.md 7)
      const int minb = mb ? atoi(mb) : 12, carve = cv ? atoi(cv) : (e->traffic_G > 0 ? (int)cudaSharedmemCarveoutMaxShared : 30);
      if (minb >= 16) return launch_mapgen_registers<RNG, 16>(e, st, grid, carve);
      if (minb >= 12) return launch_mapgen_registers<RNG, 12>(e, st, grid, carve);
      if (minb >= 10) return launch_mapgen_registers<RNG, 10>(e, st, grid, carve);
      return launch_mapgen_registers<RNG, 8>(e, st, grid, carve);
    }
  }
  auto kern = pgtg::pgtg_mapgen_kernel<RNG, TMAX, TABLED>;
  static bool carve_set = false;
  if (!carve_set) { cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); carve_set = true; }
  if (smem > 48 * 1024) { int rc = lk(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); if (rc) return rc; }
  unsigned char* const origin = (unsigned char*)4096;
  const pgtg::SharedLayout layout = pgtg::layout_of(pgtg::carve_mapgen(origin, e->dc, B), origin);
  kern<<<grid, B, smem, st>>>(e->dc, e->dp, e->dp.parity, layout);
  return lk(cudaGetLastError());
}

template <int RNG>
static int launch_mode(pgtg_env* e, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, cudaStream_t st) {
  switch (mode) {
    case MODE_STEP:
      // plain configuration: the lean instantiation (the ring-fed reset does not depend on the board size)
      if (RNG != PGTG_RNG_TAPE && e->dc.pregen && e->dc.lean && !getenv("PGTG_NO_LEAN")) {
        constexpr int R = RNG == PGTG_RNG_TAPE ? PGTG_RNG_PHILOX : RNG;
        constexpr bool L = RNG != PGTG_RNG_TAPE;  // (never launched for the tape: keeps that translation unit from instantiating it)
        if (e->dc.lean == 2) {  // sliding window and / or next_subgoal_direction
          if (e->dc.write_final_obs) return launch_one<R, MODE_STEP, 16, L, L, L, L>(e, mask, seeds, actions, action_bytes, st);
          return launch_one<R, MODE_STEP, 16, L, L, false, L>(e, mask, seeds, actions, action_bytes, st);
        }
        if (e->dc.write_final_obs) return launch_one<R, MODE_STEP, 16, L, L, L>(e, mask, seeds, actions, action_bytes, st);
        if constexpr (RNG == PGTG_RNG_PHILOX) { if (inline_mapgen_now(e)) return launch_one<R, MODE_STEP, 16, L, L, false, false, L>(e, mask, seeds, actions, action_bytes, st); }
        return launch_one<R, MODE_STEP, 16, L, L>(e, mask, seeds, actions, action_bytes, st);
      }
      if (RNG != PGTG_RNG_TAPE && e->dc.pregen) return launch_sized<RNG, MODE_STEP, RNG != PGTG_RNG_TAPE>(e, mask, seeds, actions, action_bytes, st);
      return launch_sized<RNG, MODE_STEP, false>(e, mask, seeds, actions, action_bytes, st);
    case MODE_RESET:
      return launch_sized<RNG, MODE_RESET, false>(e, mask, seeds, actions, action_bytes, st);
    case MODE_MAPGEN:
      if (RNG == PGTG_RNG_TAPE) return (int)cudaErrorInvalidValue;
      if (e->dc.conn_bits && e->dc.path_tab && !getenv("PGTG_NO_TABLED")) return launch_mapgen<RNG == PGTG_RNG_TAPE ? PGTG_RNG_PHILOX : RNG, 16, true>(e, st);
      if (e->dc.T <= 16) return launch_mapgen<RNG == PGTG_RNG_TAPE ? PGTG_RNG_PHILOX : RNG, 16>(e, st);
      if (e->dc.T <= 64) return launch_mapgen<RNG == PGTG_RNG_TAPE ? PGTG_RNG_PHILOX : RNG, 64>(e, st);
      return launch_mapgen<RNG == PGTG_RNG_TAPE ? PGTG_RNG_PHILOX : RNG, 256>(e, st);
    default:
      return launch_one<PGTG_RNG_PHILOX, MODE_OBSERVE, 16, false>(e, mask, seeds, actions, action_bytes, st);
  }
}

