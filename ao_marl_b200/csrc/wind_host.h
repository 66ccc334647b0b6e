// Wind accumulator of one turbulence layer and the sub-pixel raytrace offset derived from it, shared by the host
// (atmos.cu: the common accumulators, the mirror of per-environment accumulators) and the device (wind_state_kernel).
// Plain C++ apart from the qualifiers, so that a host compiler can build it alone.
#pragma once
#include <math.h>
#include <stdlib.h>
#include <algorithm>

#ifdef __CUDACC__
#define WIND_HD __host__ __device__ __forceinline__
#else
#define WIND_HD inline
#endif

// Raytrace offset of one layer for one environment: integer part of (sensor offset + accumulator), fractional parts
// and the bilinear weights (1-fx)(1-fy), fx(1-fy), (1-fx)fy, fx fy of the four taps.  32 bytes: one record per
// (layer, environment) when the environments of a batch have their own winds.
struct WindRec {
  int ix, iy;
  float fx, fy;
  float w00, w01, w10, w11;
};

// One frame of wind along one axis (move_atmos, atmosCompass.py:158-161): accumulate the step, return the whole pixels
// to extrude (signed) and keep the fraction.
WIND_HD int wind_advance(double& acc, float delta) {
  acc += (double)delta;
  const int n = (int)acc;
  acc -= n;
  return n;
}

// Offset of the pupil on the screen for sensor offsets (xoff, yoff) and accumulators (accx, accy) -- what
// raytrace_layer of the oracle samples.
WIND_HD WindRec wind_record(float xoff, float yoff, double accx, double accy) {
  WindRec r;
  const double px = (double)xoff + accx, py = (double)yoff + accy;
  r.ix = (int)floor(px); r.iy = (int)floor(py);
  r.fx = (float)(px - r.ix); r.fy = (float)(py - r.iy);
  r.w00 = (1.f - r.fx) * (1.f - r.fy); r.w01 = r.fx * (1.f - r.fy);
  r.w10 = (1.f - r.fx) * r.fy;         r.w11 = r.fx * r.fy;
  return r;
}

// Transitions of the per-environment wind state (wind_state_kernel, wind_load_kernel and the host mirror below)
#define WIND_STEP 0      // one frame of wind: acc += delta, counts = whole pixels
#define WIND_INIT 1      // accumulators <- the layer's common ones (ax0, ay0), no extrusion
#define WIND_RESET 2     // accumulators <- 0; counts of the start-up: 2N along y, signed like the environment's x wind
#define WIND_RESET_ENVS 3  // WIND_RESET of the listed environments envs[0..K) only (aom_reset_envs); the others keep their state
#define WIND_LOAD_ENVS 4   // accumulators of the listed environments <- loaded ones (aom_load_envs), no extrusion

// One layer of a transition
struct WindLayerParams {
  const float* dx; const float* dy;      // [E] steps in pixels per frame, or null: the common cdx / cdy
  float cdx, cdy;
  double ax0, ay0;                       // WIND_INIT
  float xoff, yoff;                      // sensor offsets of the layer (aom_config.wfs_xoff / wfs_yoff)
  int n2;                                // WIND_RESET: 2 N
};

// The host mirror of one layer's per-environment accumulators ax / ay [E] through the transition `mode` that the device
// makes, with W's winds read from host arrays.  envs [K]: the listed environments of WIND_RESET_ENVS / WIND_LOAD_ENVS, and
// lx / ly [K] their loaded accumulators.  passes: the extrusion passes of the frame along x and y, the largest |whole
// pixels| over the batch (2N along y at a reset); box: the least and greatest ix, then iy, over the batch, which bound
// the pupil footprint.
inline void wind_mirror(int mode, const WindLayerParams& W, int E, double* ax, double* ay, const int* envs, int K,
                        const double* lx, const double* ly, int passes[2], int box[4]) {
  int px = 0, py = 0;
  if (mode == WIND_RESET_ENVS) {
    for (int k = 0; k < K; ++k) ax[envs[k]] = ay[envs[k]] = 0.0;
    py = W.n2;
  }
  if (mode == WIND_LOAD_ENVS)
    for (int k = 0; k < K; ++k) { ax[envs[k]] = lx[k]; ay[envs[k]] = ly[k]; }
  for (int e = 0; e < E; ++e) {
    if (mode == WIND_STEP) {
      const int nx = wind_advance(ax[e], W.dx ? W.dx[e] : W.cdx), ny = wind_advance(ay[e], W.dy ? W.dy[e] : W.cdy);
      px = std::max(px, abs(nx)); py = std::max(py, abs(ny));
    } else if (mode == WIND_INIT) {
      ax[e] = W.ax0; ay[e] = W.ay0;
    } else if (mode == WIND_RESET) {
      ax[e] = ay[e] = 0.0;
      py = W.n2;
    }
    const WindRec r = wind_record(W.xoff, W.yoff, ax[e], ay[e]);
    if (e == 0 || r.ix < box[0]) box[0] = r.ix;
    if (e == 0 || r.ix > box[1]) box[1] = r.ix;
    if (e == 0 || r.iy < box[2]) box[2] = r.iy;
    if (e == 0 || r.iy > box[3]) box[3] = r.iy;
  }
  passes[0] = px; passes[1] = py;
}
