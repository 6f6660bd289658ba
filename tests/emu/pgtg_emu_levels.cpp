// pgtg_emu_levels.cpp -- the host emulation of pgtg_emu.cpp plus the two backend calls of level sets
// (PGTG_BACKEND_LEVELS, pgtg_api_impl.hpp). TEST INFRASTRUCTURE ONLY: the CPU tests of tests/test_levels.py load
// libpgtg_emu_levels.so; the product's CUDA backend has its own kernels for both calls (pgtg_kernels.cu).
#include <stdint.h>

struct pgtg_env;
#define PGTG_BACKEND_LEVELS
static int bk_serve_levels(pgtg_env*, void*);
static int bk_levels(pgtg_env*, int32_t*, int, void*);

#include "pgtg_emu.cpp"

// the level-serving kernel's loop: one request of the queue of launch parity dp.parity at a time
static int bk_serve_levels(pgtg_env* h, void*) {
  const uint2* list = h->dp.regen_list + (size_t)h->dp.parity * 2 * h->dc.N;
  for (uint32_t i = 0; i < h->dp.regen_count[h->dp.parity]; i++) phase_serve_level(h->dc, h->dp, (int)list[i].x, list[i].y);
  return 0;
}

static int bk_levels(pgtg_env* h, int32_t* out, int previous, void*) {
  for (int env = 0; env < h->dc.N; env++) out[env] = env_level(h->dc, h->dp, env, previous);
  return 0;
}
