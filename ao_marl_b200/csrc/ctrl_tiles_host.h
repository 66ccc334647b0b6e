// Host side of the per-environment controllers (aom_set_controller_env): the tile list the per-environment form of
// actor_fused_kernel (actor_tc.cuh) runs over.  Plain C++, no CUDA, so that a host build of it
// (tests/cpu_kernels/ctrl_tiles_harness.cpp) checks the same code the library runs.
//
// A tile is one policy slot and up to CTL_TILE environment indices of that slot, -1 as padding.  The environments are
// grouped by slot (ascending), in ascending order within a slot; environments on the integrator (AOM_CTRL_INTEGRATOR)
// are left out.  The kernel's grid is (tiles, agents), so the tiles of one (slot, agent) are launched next to each other
// and a slot's weights are read from L2 by all but the first of them.
#pragma once
#include <stdint.h>
#include "../../include/aomarl.h"

#define CTL_TILE 128                      // environment rows per tile (GTC_BM of the actor kernel)

// Upper bound of the tiles of a batch of E environments: every slot may leave one partial tile
static inline int ctl_tiles_max(int E) { return (E + CTL_TILE - 1) / CTL_TILE + AOM_MAX_POLICIES; }

// ctrl [E]: a slot 0 .. AOM_MAX_POLICIES-1 or AOM_CTRL_INTEGRATOR per environment (checked by the caller).  Fills
// tile_slot [n] and tile_env [n][CTL_TILE] for the n <= ctl_tiles_max(E) tiles and returns n; integ [E] receives the
// environments on the integrator, their count in *n_integ.
static inline int ctl_build_tiles(const int32_t* ctrl, int E, int32_t* tile_slot, int32_t* tile_env, int32_t* integ,
                                  int* n_integ) {
  int n = 0, ni = 0;
  for (int s = 0; s < AOM_MAX_POLICIES; ++s) {
    int r = CTL_TILE;                                   // rows used in tile n - 1
    for (int e = 0; e < E; ++e) {
      if (ctrl[e] != s) continue;
      if (r == CTL_TILE) {
        tile_slot[n] = s;
        for (int i = 0; i < CTL_TILE; ++i) tile_env[(size_t)n * CTL_TILE + i] = -1;
        ++n;
        r = 0;
      }
      tile_env[(size_t)(n - 1) * CTL_TILE + r++] = e;
    }
  }
  for (int e = 0; e < E; ++e)
    if (ctrl[e] == AOM_CTRL_INTEGRATOR) integ[ni++] = e;
  *n_integ = ni;
  return n;
}
