// Host interface of the turbulence layers (atmos.cu): the screens with their ring origins and extrusion counters, the
// wind state -- common accumulators, or per environment on the device with a host mirror -- and the extrusion that
// moves the screens with it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/aomarl.h"
#include "env_cond.h"
#include "wfs_params.cuh"

struct Atmos;

// What the atmosphere reads from its context on every call; each pointer stays valid for the context's life.
struct AtmosLinks {
  const EnvCond (*cond)[AOM_MAX_LAYERS];   // the conditions [aom_condition][layer]: amplitudes and winds
  void* const (*tab)[AOM_MAX_LAYERS];      // the device tables [aom_table][index]: AB and stencil of each layer
  const int* opt;                          // the options [aom_option]: extrusion path, GEMM path
  const uint32_t* k0;                      // Philox keys [E]
  const uint32_t* k1;
  int* err_word;                           // device error word raised by bounded waits
  uint64_t* launches;                      // the context's count of kernel launches
  int num_sms;
};

// The device buffers of one layer, each [E] rows: screen [E][N][N], ring origins, extrusions done since reset
struct AtmosLayer {
  float* screen;
  int* ox;
  int* oy;
  uint32_t* count;
};

// Every function returns AOM_OK, or an error code with its message in err.  *out is set even on failure, for
// atmos_destroy.
int atmos_create(const aom_config& c, const AtmosLinks& links, Atmos** out, char (&err)[512]);
void atmos_destroy(Atmos* a);

AtmosLayer atmos_layer(const Atmos* a, int l);

// Takes note of an uploaded table (aom_set_table), before the context keeps it: the digit planes of a layer's [A | B]
// for the integer extrusion.  A non-finite operator is refused and changes nothing.
int atmos_set_table(Atmos* a, int table, int index, const void* host, char (&err)[512]);

// New screens for every environment (aom_reset, after the keys), or for the K environments listed in envs_d (device) /
// envs_h (host) (aom_reset_envs, after their keys, screens, ring origins and counters were cleared).
int atmos_reset(Atmos* a, cudaStream_t st, char (&err)[512]);
int atmos_reset_envs(Atmos* a, const int* envs_d, const int* envs_h, int K, cudaStream_t st, char (&err)[512]);

// One frame of wind: every layer extrudes the whole pixels its accumulators crossed (aom_move_atmos)
int atmos_move(Atmos* a, cudaStream_t st, char (&err)[512]);

// After a change of the per-environment winds of `layer`: the common state when it can, else every environment continues
// from the common accumulators (the screens do not jump), and its pupil footprint must stay on the screen.
int atmos_settle(Atmos* a, int layer, char (&err)[512]);

// The wind accumulators of n loaded records h (aom_load_envs) for the environments listed in envs_d / envs_h.  stage:
// host room for 2 L n doubles, which the stream may read until the call returns.
int atmos_load(Atmos* a, int n, const int* envs_d, const int* envs_h, const aom_env_head* h, double* stage,
               cudaStream_t st, char (&err)[512]);

// The layers of a sampler's frame, p.layer[0..p.n_layers), and its per-environment offsets p.wind; refused when the pupil
// footprint leaves a screen.
int atmos_fill_layers(const Atmos* a, WfsParams& p, char (&err)[512]);

// What a record keeps of the wind state (aom_save_envs): the common accumulators acc[l] = (x, y), and the per-environment
// ones [L][2][E] on the device, or null while the common ones are in force.
const double* atmos_snap_view(const Atmos* a, double (*acc)[2]);
