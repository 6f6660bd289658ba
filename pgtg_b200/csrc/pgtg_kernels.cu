// pgtg_kernels.cu -- sm_100a kernels and the CUDA backend of the C ABI (include/pgtg_b200.h).
//
// One fused launch per tick: every CTA owns a contiguous slice of B envs and runs
//   stage -> step (1 env / thread) -> ballot+scan compaction of done envs -> on-device reset /
//   procedural map regeneration by the first n_done threads -> observation bit assembly in shared
//   memory -> vectorised expansion to the int8 observation planes (contiguous 16-byte stores).
// Nothing here is a dense contraction, so no tensor cores: the kernel is bounded by HBM traffic
// (observation write + SoA state scan), see DESIGN.md for the byte accounting.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "pgtg_phases.cuh"

struct pgtg_env;
static thread_local cudaError_t g_cuda_err = cudaSuccess;
static const char* bk_error() { return cudaGetErrorString(g_cuda_err); }
static int ck(cudaError_t e) { if (e != cudaSuccess) { g_cuda_err = e; return -1; } return 0; }
static void* bk_alloc(size_t n) { void* p = nullptr; if (ck(cudaMalloc(&p, n))) return nullptr; return p; }
static void bk_free(void* p) { cudaFree(p); }
static int bk_set_device(int d) { return ck(cudaSetDevice(d)); }
static int bk_h2d(void* d, const void* s, size_t n, void* st) { return ck(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, (cudaStream_t)st)); }
static int bk_d2h(void* d, const void* s, size_t n, void* st) { return ck(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, (cudaStream_t)st)); }
static int bk_d2d(void* d, const void* s, size_t n, void* st) { return ck(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, (cudaStream_t)st)); }
static void* bk_stream_create() { cudaStream_t s; if (ck(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking))) return nullptr; return s; }
static void bk_stream_destroy(void* s) { cudaStreamDestroy((cudaStream_t)s); }
static int bk_memset(void* d, int v, size_t n) { return ck(cudaMemset(d, v, n)); }
static int bk_memset_async(void* d, int v, size_t n, void* st) { return ck(cudaMemsetAsync(d, v, n, (cudaStream_t)st)); }
static int bk_sync(void* st) { return ck(st ? cudaStreamSynchronize((cudaStream_t)st) : cudaDeviceSynchronize()); }
// side stream (highest priority) for the persistent map-generation kernel, and its events
static int bk_side_create(void** stream, void** ev_tick, void** ev_map0, void** ev_map1, int* sm_count) {
  int lo = 0, hi = 0, dev = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
  cudaStream_t s; cudaEvent_t a, b, c;
  if (ck(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi))) return -1;  // priority made no measurable difference
  if (ck(cudaEventCreateWithFlags(&a, cudaEventDisableTiming)) || ck(cudaEventCreateWithFlags(&b, cudaEventDisableTiming)) ||
      ck(cudaEventCreateWithFlags(&c, cudaEventDisableTiming))) return -1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev);
  *stream = s; *ev_tick = a; *ev_map0 = b; *ev_map1 = c;
  return 0;
}
static void bk_side_destroy(void* stream, void* a, void* b, void* c) {
  if (stream) { cudaStreamSynchronize((cudaStream_t)stream); cudaStreamDestroy((cudaStream_t)stream); }
  if (a) cudaEventDestroy((cudaEvent_t)a);
  if (b) cudaEventDestroy((cudaEvent_t)b);
  if (c) cudaEventDestroy((cudaEvent_t)c);
}
static int bk_stream_wait(void* st, void* ev) { return ck(cudaStreamWaitEvent((cudaStream_t)st, (cudaEvent_t)ev, 0)); }
static int bk_dl_device_type() { return 2; }  // kDLCUDA
static void* bk_event_create() { cudaEvent_t ev; if (ck(cudaEventCreate(&ev))) return nullptr; return ev; }
static void bk_event_destroy(void* ev) { cudaEventDestroy((cudaEvent_t)ev); }
static int bk_event_record(void* ev, void* st) { return ck(cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)st)); }
static double bk_event_elapsed(void* a, void* b) { float ms = 0; cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b); return ms; }
static int bk_launch(pgtg_env*, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream);
static int bk_stats_reduce(pgtg_env*, void* stream);
static int bk_stats_reset(pgtg_env*, void* stream);
static int bk_flatten(pgtg_env*, void* stream);
static int bk_info(pgtg_env*, int32_t* out_dev);
static int bk_error_or(pgtg_env*, uint32_t* out_dev);
#define PGTG_BACKEND_LEVELS
static int bk_serve_levels(pgtg_env*, void* stream);
static int bk_levels(pgtg_env*, int32_t* out_dev, int previous, void* stream);
#define PGTG_BACKEND_OBS_BITS
static int bk_unpack_bits(pgtg_env*, const pgtg::UnpackArgs& a, int format, void* out_dev, const int* plane_order, void* stream);
static int bk_conn_table_max_bits() { return 24; }
static bool bk_inline_mapgen() { return true; }
static int bk_build_conn_table(pgtg_env*, uint32_t* table_dev);
static int bk_build_path_table(pgtg_env*, uint64_t* table_dev);
int pgtg_traffic_geometry(const pgtg::DevCfg& c, int* G, int* NT, size_t* smem);  // pgtg_traffic.cu
static void bk_traffic_geometry(const pgtg::DevCfg& c, int* G, int* NT) { size_t smem; pgtg_traffic_geometry(c, G, NT, &smem); }

#include "pgtg_api_impl.hpp"

namespace pgtg {

// one thread per 32-bit word of the start-goal connectivity table (32 subgraphs each)
__global__ void pgtg_build_conn_table_kernel(const __grid_constant__ DevCfg c, uint32_t* __restrict__ table, int s, int g) {
  const uint32_t words = (1u << c.conn_bits) / 32u + ((1u << c.conn_bits) < 32u ? 1u : 0u);
  const uint32_t rowmask = (1u << (c.W - 1)) - 1u, emask = (1u << c.conn_ne) - 1u;
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += gridDim.x * blockDim.x) {
    uint32_t bits = 0;
    for (uint32_t b = 0; b < 32; b++) {
      uint32_t idx = w * 32u + b, ec = idx & emask, so = idx >> c.conn_ne, e = 0;
      for (int r = 0; r < c.H; r++) e |= ((ec >> (r * (c.W - 1))) & rowmask) << (r * c.W);
      if (flood_connected32(c.W, e, so, s, g)) bits |= 1u << b;
    }
    table[w] = bits;
  }
}

struct FlatOrder { int plane[PGTG_MAX_CHANNELS]; };

__global__ void pgtg_error_or_kernel(const uint32_t* __restrict__ err, int n, uint32_t* __restrict__ out) {
  uint32_t v = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) v |= err[i];
  v = __reduce_or_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicOr(out, v);
}

// get_info extras, one env per thread (tile descriptors read straight from HBM)
__global__ void __launch_bounds__(128) pgtg_info_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, int32_t* __restrict__ out) {
  __shared__ __align__(16) Lut lut;
  BlockShared sh;
  sh.lut = &lut;
  stage_tables(c, p, sh, threadIdx.x, blockDim.x, false);
  __syncthreads();
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env < c.N) info_env(c, p, lut, env, out);
}

// one thread per entry of the subgoal-path table
__global__ void __launch_bounds__(128) pgtg_build_path_table_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, uint64_t* __restrict__ table) {
  extern __shared__ __align__(16) unsigned char smem[];
  BlockShared sh = carve_mapgen(smem, c, blockDim.x);
  stage_tables(c, p, sh, threadIdx.x, blockDim.x);
  __syncthreads();
  const uint32_t total = 1u << c.conn_bits;
  for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x)
    table[g] = path_table_entry(c, *sh.lut, g, sh.tiles + threadIdx.x * c.tile_stride);
}

// FlattenObservation view: one warp per env; the C*P*P plane cells are one flat index space (cell -> plane by a multiply-high,
// no division), a lane takes eight cells 32 apart per round and issues the eight byte loads before the first store, so a
// warp keeps eight sectors in flight instead of one (the one-load-at-a-time loop this replaces was bound by that latency:
// 0.51 ms for 262 144 envs of the train.py configuration; now 0.33 ms = 4.3 TB/s of reads + float32 stores, 66 % of the
// measured HBM bandwidth). Measured and no faster: sixteen loads per round, a plane-uniform chunk loop, reading the packed
// bits instead of the int8 planes -- what is left is the 4.5 KB of 32-bit stores per env. Reads go through L2.
__global__ void __launch_bounds__(256) pgtg_flatten_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, const __grid_constant__ FlatOrder order,
                                                          float* __restrict__ out, int dim, uint32_t inv_pp /* ceil(2^32 / (P*P)) */) {
  const int PP = c.P * c.P, total = c.C * PP, lane = threadIdx.x & 31;
  for (int env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); env < c.N; env += gridDim.x * (blockDim.x >> 5)) {
    float* o = out + (size_t)env * dim;
    const int8_t* m = p.obs_map + (size_t)env * total;
    for (int base = lane; base < total; base += 32 * 8) {
      int8_t v[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int idx = base + 32 * u;
        v[u] = 0;
        if (idx < total) {
          const int k = PP == 1 ? idx : (int)__umulhi((uint32_t)idx, inv_pp);  // idx / PP (exact: idx < 2^16; 2^32 / 1 does not fit)
          v[u] = __ldg(m + order.plane[k] * PP + (idx - k * PP));
        }
      }
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int idx = base + 32 * u;
        if (idx < total) o[idx] = (float)v[u];
      }
    }
    o += total;
    if (c.use_nsd) {  // Discrete(9, start=-1) one-hot
      if (lane < 9) o[lane] = (p.obs_nsd[env] + 1 == lane) ? 1.0f : 0.0f;
      o += 9;
    }
    if (lane < 18) o[lane] = (p.obs_position[2 * env + (lane >= 9)] == (lane >= 9 ? lane - 9 : lane)) ? 1.0f : 0.0f;  // MultiDiscrete([9, 9]) -> two one-hots
    else if (lane < 20) o[lane] = (float)p.obs_velocity[2 * env + (lane - 18)];
  }
}

// Level sets: the map-generation launch of the pipeline replaced by copies from the pool (phase_serve_level), dense over the
// same request queue, one request per thread, grid-stride like the generator so that the persistent-grid option applies.
__global__ void __launch_bounds__(128) pgtg_serve_levels_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, int parity) {
  const uint32_t count = p.regen_count[parity];
  const uint2* list = p.regen_list + (size_t)parity * 2 * c.N;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint2 r = list[i];
    phase_serve_level(c, p, (int)r.x, r.y);
  }
}

// pgtg_levels: every env's level, recomputed from its key and episode counter
__global__ void __launch_bounds__(256) pgtg_levels_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ DevPtrs p, int previous, int32_t* __restrict__ out) {
  for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < c.N; env += gridDim.x * blockDim.x) out[env] = env_level(c, p, env, previous);
}

// pgtg_unpack_bits, int8 format: one thread per 32 output cells (unpack_chunk), expanded with the tick's byte -> 8 cells table and
// stored as one 256-bit vector, consecutive threads -> consecutive vectors (the output is 32-byte aligned)
__global__ void __launch_bounds__(256) pgtg_unpack_int8_kernel(const UnpackArgs a, int obs_bits, int8_t* __restrict__ out) {
  __shared__ uint2 lut[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) { uint2 v; v.x = spread4((uint32_t)i); v.y = spread4((uint32_t)i >> 4); lut[i] = v; }
  __syncthreads();
  const uint64_t total = (uint64_t)a.count * (uint64_t)obs_bits, n32 = total / 32u, nchunks = (total + 31u) / 32u;
  bool bad = false;
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < nchunks; j += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t w = unpack_chunk(a, obs_bits, j, &bad);
    if (j < n32) pg_store_streaming32(out + 32u * j, lut[w & 255u], lut[(w >> 8) & 255u], lut[(w >> 16) & 255u], lut[w >> 24]);
    else for (uint64_t b = 32u * j; b < total; b++) out[b] = (int8_t)((w >> (uint32_t)(b - 32u * j)) & 1u);
  }
  if (bad) atomicOr(a.err, PGTG_UNPACK_INDEX_ERROR);
}

// pgtg_unpack_bits, flat format: one warp per output row, the planes in sorted-key order (a lane per cell), then the scalars
__global__ void __launch_bounds__(256) pgtg_unpack_flat_kernel(const __grid_constant__ DevCfg c, const UnpackArgs a, const __grid_constant__ FlatOrder order,
                                                              float* __restrict__ out, int dim) {
  const int lane = threadIdx.x & 31, PP = c.P * c.P;
  bool bad = false;
  for (int64_t o = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); o < a.count; o += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    const int64_t r = unpack_source_row(a, o);
    bad |= r < 0;
    const uint64_t bit0 = r >= 0 ? unpack_row_bit0(a, c.obs_bits, r) : 0u;
    float* row = out + o * dim;
    for (int k = 0; k < c.C; k++)
      for (int cell = lane; cell < PP; cell += 32) row[k * PP + cell] = unpack_flat_cell(c, a, order.plane, r, bit0, k, cell);
    for (int q = lane; q < dim - c.C * PP; q += 32) row[c.C * PP + q] = unpack_flat_tail(c, a, r, q);
  }
  if (bad && lane == 0) atomicOr(a.err, PGTG_UNPACK_INDEX_ERROR);
}

__global__ void pgtg_reduce_stats_kernel(const double* __restrict__ rows, int nrows, double* __restrict__ out) {
  // out[k] = sum over CTAs of rows[.][k]; one warp per statistic
  int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double s = 0;
  for (int r = lane; r < nrows; r += 32) s += rows[(size_t)r * STATS_STRIDE + k];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) out[k] = s;
}

}  // namespace pgtg

// ---- CUDA backend: launch ----------------------------------------------------------------------
// the kernel instantiations live in pgtg_inst_*.cu (one per random-number source); they return the cudaError_t
int pgtg_launch_mode_philox(pgtg_env*, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream);
int pgtg_launch_mode_tape(pgtg_env*, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream);
int pgtg_launch_mode_numpy(pgtg_env*, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream);

int pgtg_launch_traffic_tick(pgtg_env* e, const void* actions, int action_bytes, void* stream);  // pgtg_traffic.cu

static int bk_launch(pgtg_env* e, int mode, const uint8_t* mask, const int64_t* seeds, const void* actions, int action_bytes, void* stream) {
  // configurations with cars (Philox mode): the traffic tick; reset / observe stay on the general kernel
  if (mode == MODE_STEP && e->traffic_G > 0) return ck((cudaError_t)pgtg_launch_traffic_tick(e, actions, action_bytes, stream));
  switch (e->cfg.rng_mode) {
    case PGTG_RNG_TAPE: return ck((cudaError_t)pgtg_launch_mode_tape(e, mode, mask, seeds, actions, action_bytes, stream));
    case PGTG_RNG_NUMPY: return ck((cudaError_t)pgtg_launch_mode_numpy(e, mode, mask, seeds, actions, action_bytes, stream));
    default: return ck((cudaError_t)pgtg_launch_mode_philox(e, mode, mask, seeds, actions, action_bytes, stream));
  }
}

extern "C" int pgtg_observe(pgtg_env* e, void* stream) {
  if (!e || !e->did_reset) return fail(PGTG_ERR_STATE, "observe before reset");
  bk_set_device(e->device);
  if (bk_launch(e, MODE_OBSERVE, nullptr, nullptr, nullptr, 0, stream)) return fail(PGTG_ERR_CUDA, std::string("observe launch failed: ") + bk_error());
  e->launches++;
  return PGTG_OK;
}

// Sum the per-CTA statistic rows into the 8-double `stats` buffer on the device (the buffer the
// host all-reduces with NCCL), on `stream`, without synchronising.
static int bk_stats_reduce(pgtg_env* e, void* stream) {
  pgtg::pgtg_reduce_stats_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(e->stats_rows, e->stats_nrows, e->dp.stats);
  e->launches++;
  return ck(cudaGetLastError());
}
static int bk_build_conn_table(pgtg_env* e, uint32_t* table_dev) {
  int s = e->dc.start_y * e->dc.W + e->dc.start_x, g = e->dc.goal_y * e->dc.W + e->dc.goal_x;
  pgtg::pgtg_build_conn_table_kernel<<<148 * 8, 256>>>(e->dc, table_dev, s, g);
  return ck(cudaGetLastError());
}
static int bk_build_path_table(pgtg_env* e, uint64_t* table_dev) {
  const int B = 128;
  size_t smem = pgtg::mapgen_shared_bytes(e->dc, B);
  uint32_t total = 1u << e->dc.conn_bits;
  int blocks = (int)((total + B - 1) / B < 148u * 12u ? (total + B - 1) / B : 148u * 12u);
  pgtg::pgtg_build_path_table_kernel<<<blocks, B, smem>>>(e->dc, e->dp, table_dev);
  return ck(cudaGetLastError());
}
static int bk_error_or(pgtg_env* e, uint32_t* out_dev) {
  if (ck(cudaMemsetAsync(out_dev, 0, 4, nullptr))) return -1;
  pgtg::pgtg_error_or_kernel<<<148 * 4, 256>>>(e->dp.error, e->dc.N, out_dev);
  return ck(cudaGetLastError());
}
static int bk_info(pgtg_env* e, int32_t* out_dev) {
  pgtg::pgtg_info_kernel<<<(e->dc.N + 127) / 128, 128>>>(e->dc, e->dp, out_dev);
  return ck(cudaGetLastError());
}
static int bk_flatten(pgtg_env* e, void* stream) {
  pgtg::FlatOrder order;
  for (int i = 0; i < PGTG_MAX_CHANNELS; i++) order.plane[i] = e->flat_order[i];
  const int warps = 8, want = (e->dc.N + warps - 1) / warps;
  const int blocks = want < 148 * 32 ? want : 148 * 32;
  const uint32_t pp = (uint32_t)(e->dc.P * e->dc.P), inv_pp = (uint32_t)((0x100000000ull + pp - 1) / pp);
  pgtg::pgtg_flatten_kernel<<<blocks, 32 * warps, 0, (cudaStream_t)stream>>>(e->dc, e->dp, order, e->flat, e->flat_dim, inv_pp);
  return ck(cudaGetLastError());
}
static int bk_serve_levels(pgtg_env* e, void* stream) {
  const int full = (2 * e->dc.N + 127) / 128, grid = e->mapgen_grid > 0 && e->mapgen_grid < full ? e->mapgen_grid : full;
  pgtg::pgtg_serve_levels_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(e->dc, e->dp, e->dp.parity);
  return ck(cudaGetLastError());
}
static int bk_levels(pgtg_env* e, int32_t* out_dev, int previous, void* stream) {
  const int blocks = (e->dc.N + 255) / 256;
  pgtg::pgtg_levels_kernel<<<blocks < 148 * 8 ? blocks : 148 * 8, 256, 0, (cudaStream_t)stream>>>(e->dc, e->dp, previous, out_dev);
  return ck(cudaGetLastError());
}
static int bk_unpack_bits(pgtg_env* e, const pgtg::UnpackArgs& a, int format, void* out_dev, const int* plane_order, void* stream) {
  if (a.count == 0) return 0;
  if (format == PGTG_UNPACK_INT8) {
    const uint64_t chunks = ((uint64_t)a.count * (uint64_t)e->dc.obs_bits + 31u) / 32u, want = (chunks + 255u) / 256u;
    if (!chunks) return 0;
    pgtg::pgtg_unpack_int8_kernel<<<(int)(want < 148u * 16u ? want : 148u * 16u), 256, 0, (cudaStream_t)stream>>>(a, e->dc.obs_bits, (int8_t*)out_dev);
  } else {
    pgtg::FlatOrder order;
    for (int i = 0; i < PGTG_MAX_CHANNELS; i++) order.plane[i] = i < e->dc.C ? plane_order[i] : 0;
    const int64_t want = (a.count + 7) / 8;
    pgtg::pgtg_unpack_flat_kernel<<<(int)(want < 148 * 32 ? want : 148 * 32), 256, 0, (cudaStream_t)stream>>>(e->dc, a, order, (float*)out_dev, pgtg::unpack_flat_dim(e->dc));
  }
  return ck(cudaGetLastError());
}
static int bk_stats_reset(pgtg_env* e, void* stream) {
  if (ck(cudaMemsetAsync(e->stats_rows, 0, sizeof(double) * pgtg::STATS_STRIDE * (size_t)e->stats_nrows, (cudaStream_t)stream))) return -1;
  return ck(cudaMemsetAsync(e->dp.stats, 0, 64, (cudaStream_t)stream));
}
