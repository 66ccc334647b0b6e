// Host build of ctrl_tiles_host.h, the tile list the per-environment actor kernel runs over (aom_set_controller_env), so
// that the exact code the library runs is checked on a machine without a GPU.
// Built by tests/test_controller_tiles.py:  g++ -O2 -shared -fPIC
#include <cstdint>
#include "../../ao_marl_b200/csrc/ctrl_tiles_host.h"

extern "C" {

int h_ctrl_tiles_max(int E) { return ctl_tiles_max(E); }

// Returns the tile count; fills tile_slot [n], tile_env [n][CTL_TILE], integ [*n_integ]
int h_ctrl_tiles(const int32_t* ctrl, int E, int32_t* tile_slot, int32_t* tile_env, int32_t* integ, int* n_integ) {
  return ctl_build_tiles(ctrl, E, tile_slot, tile_env, integ, n_integ);
}
}
