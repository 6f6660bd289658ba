// pgtg_env.hpp -- the native handle behind the C ABI (include/pgtg_b200.h): configuration, device pointers,
// launch geometry and the map-generation pipeline state. Shared by the API implementation
// (pgtg_api_impl.hpp) and by the translation units that hold the kernel instantiations.
#pragma once
#include <stdint.h>

#include <vector>

#include "pgtg_phases.cuh"

using namespace pgtg;

namespace pgtg { constexpr int STATS_STRIDE = 8; }  // doubles per per-CTA episode-statistics row

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_OBSERVE = 2, MODE_MAPGEN = 3 };

struct pgtg_env {
  pgtg_config cfg;
  DevCfg dc;
  DevPtrs dp;
  int device;
  int block;
  size_t smem;
  int64_t launches;
  std::vector<void*> allocs;
  struct StateAlloc { void* ptr; size_t bytes; };
  std::vector<StateAlloc> state_allocs;  // everything pgtg_save_state / pgtg_copy_state must carry (SoA state, rings, queues, outputs)
  bool have_fixed, have_tape, did_reset;
  int max_steps_cfg;    // episode cap of the configuration (or adopted by pgtg_copy_state); dc.max_episode_steps is the cap in force
  int gamma_cap;        // entries of dp.gamma_pow (pgtg_set_evaluation reuses the table while max_steps fits)
  bool cars_injected;   // pgtg_set_state put cars into the handle: the lean tick is off for good
  int nblk;             // CTAs per launch
  int stats_nrows;      // rows of stats_rows (one per CTA of the kernel with the most CTAs)
  int traffic_G, traffic_NT;  // geometry of the traffic tick (pgtg_traffic.cu); G = 0: not used for this handle
  // pregen pipeline: the persistent map-generation kernel runs on a side stream and overlaps the next tick
  void* side_stream; void* ev_tick; void* ev_map[2];
  uint64_t launch_index;
  bool inline_mapgen;   // experiment (PGTG_INLINE_MAPGEN): the lean tick rebuilds consumed ring slots itself
  int mapgen_grid;      // CTAs of the persistent map-generation kernel (0 = one per 128 requests)
  int mapgen_grid_overlap; bool overlap;  // overlap on: side stream + small grid; off: same stream, full grid
  // optional per-kernel timing (CUDA events on the launching stream around each kernel of a tick)
  bool timing; std::vector<void*> tev; int tev_used;
  // flattened observation (FlattenObservation view for SB3-style consumers), allocated on first use
  float* flat; int flat_dim; int flat_order[PGTG_MAX_CHANNELS];
  // host-buffer steps: packed observation bits + staging for the double-buffered copies (allocated on first use)
  uint32_t* packed_dev; unsigned char* stage_dev[2]; size_t stage_bytes; void* copy_stream; void* ev_stage[2]; void* ev_copied[2]; uint64_t host_steps;
  // observation format (pgtg_set_obs_format): in bits mode dp.obs_map / dp.f_obs_map are null and the int8 buffers live here,
  // written by pgtg_expand_obs only; the bits buffers are state allocations
  int obs_format; int8_t* obs_map_buf; int8_t* f_obs_map_buf; uint32_t* obs_packed_buf; uint32_t* f_obs_packed_buf;
  uint32_t* unpack_err;  // device word: error flag 256 of pgtg_unpack_bits (pgtg_error_summary)
  int32_t* info_dev;    // [7][N] scratch of pgtg_get_info, allocated on first use
  double* stats_rows;   // [nblk][8] per-CTA episode statistics (CUDA backend)
  // device scratch for reset arguments and host-buffer steps
  uint8_t* mask_dev;
  int64_t* seeds_dev;
  int32_t* actions_dev;
  // host tables kept for get_state / introspection
  std::vector<uint16_t> edge_tab, edge_rev, border_slots;
};

// the lean tick generates the maps itself (experiment, PGTG_INLINE_MAPGEN): plain lean configuration only
static inline bool inline_mapgen_now(const pgtg_env* e) { return e->inline_mapgen && e->dc.pregen && e->dc.lean == 1 && !e->dc.write_final_obs; }
