// pgtg_emu_bits.cpp -- the host emulation of pgtg_emu_levels.cpp plus the bits observation format (PGTG_BACKEND_OBS_BITS,
// pgtg_api_impl.hpp): the unpack backend call, and the terminal observations stored as words. TEST INFRASTRUCTURE ONLY: the
// CPU tests of tests/test_obs_bits.py load libpgtg_emu_bits.so; the product's CUDA backend has its own unpack kernels
// (pgtg_kernels.cu) and passes final_obs_packed to the phases itself.
#include <stdint.h>

#include "../../pgtg_b200/csrc/pgtg_phases.cuh"

struct pgtg_env;
#define PGTG_BACKEND_OBS_BITS
static int bk_unpack_bits(pgtg_env*, const pgtg::UnpackArgs&, int, void*, const int*, void*);

// The emulated CTA loops of pgtg_emu.cpp name only the int8 destination of the terminal observations, which is null in bits
// mode; hand the phases the words' destination and the CTA's env count as the tick kernels do (`p` and `nvalid` are the loops'
// own). The phases are defined above, so only the calls below are rewritten.
#define phase_expand_final_vec(c, out, sh, t, B, env0, nvalid, words) phase_expand_final_vec(c, out, sh, t, B, env0, nvalid, words, p.f_obs_packed)
#define phase_expand_final(c, out, sh, t, B, env0, n_done) phase_expand_final(c, out, sh, t, B, env0, n_done, p.f_obs_packed, nvalid)

#include "pgtg_emu_levels.cpp"

#undef phase_expand_final_vec
#undef phase_expand_final

// the unpack kernels' loops: one 32-cell chunk (int8) or one output row (flat) at a time
static int bk_unpack_bits(pgtg_env* h, const UnpackArgs& a, int format, void* out, const int* order, void*) {
  const DevCfg& c = h->dc;
  bool bad = false;
  if (format == PGTG_UNPACK_INT8) {
    const uint64_t total = (uint64_t)a.count * (uint64_t)c.obs_bits;
    int8_t* o = (int8_t*)out;
    for (uint64_t j = 0; j < (total + 31) / 32; j++) {
      const uint32_t w = unpack_chunk(a, c.obs_bits, j, &bad);
      for (uint64_t b = 32 * j; b < total && b < 32 * j + 32; b++) o[b] = (int8_t)((w >> (uint32_t)(b - 32 * j)) & 1u);
    }
  } else {
    const int PP = c.P * c.P, dim = unpack_flat_dim(c);
    for (int64_t row = 0; row < a.count; row++) {
      const int64_t r = unpack_source_row(a, row);
      bad |= r < 0;
      const uint64_t bit0 = r >= 0 ? unpack_row_bit0(a, c.obs_bits, r) : 0u;
      float* o = (float*)out + row * dim;
      for (int k = 0; k < c.C; k++)
        for (int cell = 0; cell < PP; cell++) o[k * PP + cell] = unpack_flat_cell(c, a, order, r, bit0, k, cell);
      for (int q = 0; q < dim - c.C * PP; q++) o[c.C * PP + q] = unpack_flat_tail(c, a, r, q);
    }
  }
  if (bad) *a.err |= PGTG_UNPACK_INDEX_ERROR;
  return 0;
}
