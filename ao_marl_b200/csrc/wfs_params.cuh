// Parameter blocks shared by every Shack-Hartmann frame kernel (wfs_kernels.cuh, wfs_mma.cuh, wfs_tma.cuh,
// wfs_umma.cuh): one turbulence layer as the raytrace sees it, and the per-frame sensor / mirror description.
#pragma once
#include <stdint.h>
#include "../../include/aomarl.h"
#include "wind_host.h"

struct WfsLayer {
  const float* screen;   // [E][N][N]
  const int* ox; const int* oy;
  int N;
  int ix, iy;            // integer part of (offset + wind accumulator)
  float fx, fy;          // fractional part
  float w00, w01, w10, w11;   // bilinear weights (1-fx)(1-fy), fx(1-fy), (1-fx)fy, fx fy of the four taps
};

struct WfsParams {
  WfsLayer layer[AOM_MAX_LAYERS];
  int n_layers;          // 0 when the atmosphere is not traced
  int use_dm;
  int E, n, nvalid;
  const float* mpupil;   // [n][n]
  const float* halfxy;   // [16][16]
  const int* sub_x0; const int* sub_y0; const float* flux;
  // mirrors
  const float* volts; int ldv;         // [E][ldv]: pzt volts then 2 tip-tilt volts
  const float* stamp1d; int ss;
  const int* act_map; int grid_n, pitch, i1_0, j1_0, pzt_off, pzt_nact;
  const float* tt_planes; int tt_dim, tt_off;
  // sensor
  float k2;              // 2 pi / lambda
  float nphotons, noise;
  float cog_offset, pixsize;
  uint32_t frame, wfs_index;
  const uint32_t* k0; const uint32_t* k1;
  const uint32_t* frame0;              // [E] or null: environment e's noise frame is frame - frame0[e] (aom_reset_envs)
  // outputs
  float* slopes; int lds;              // [E][lds]: x slopes then y slopes
  float* bincube;                      // [E][nvalid][256] or null
  // per-environment winds: offsets of every layer and environment [n_layers][E], read by the kernels' per-environment
  // instantiations in place of layer[l].ix .. w11 (null while every layer moves all environments alike)
  const WindRec* wind;
  // per-environment sensor values [E] (aom_set_wfs_noise_env), read by the kernels' NE instantiations in place of noise /
  // nphotons (null: the common value; noise_env is null in a frame drawn noise-free)
  const float* noise_env;
  const float* nph_env;
};

// sensor noise / photon count of environment e: the common value, or its own when NE (per-environment sensor values)
template <bool NE>
__device__ __forceinline__ float noise_of(const WfsParams& p, int e) {
  return (NE && p.noise_env) ? p.noise_env[e] : p.noise;
}
template <bool NE>
__device__ __forceinline__ float nphotons_of(const WfsParams& p, int e) {
  return (NE && p.nph_env) ? p.nph_env[e] : p.nphotons;
}

// raytrace offset of layer l for environment e: the layer's common one, or its record when PE (per-environment winds)
template <bool PE>
__device__ __forceinline__ WindRec wind_of(const WfsParams& p, int l, int e) {
  if (PE) return p.wind[(size_t)l * p.E + e];
  const WfsLayer& L = p.layer[l];
  WindRec r;
  r.ix = L.ix; r.iy = L.iy; r.fx = L.fx; r.fy = L.fy; r.w00 = L.w00; r.w01 = L.w01; r.w10 = L.w10; r.w11 = L.w11;
  return r;
}

// noise frame of environment e: its frames count from its own reset once environments are staggered
__device__ __forceinline__ uint32_t noise_frame(const WfsParams& p, int e) {
  return p.frame0 ? p.frame - p.frame0[e] : p.frame;
}

