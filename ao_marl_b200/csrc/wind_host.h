// Wind accumulator of one turbulence layer and the sub-pixel raytrace offset derived from it, shared by the host
// (aom_move_atmos, fill_wfs_params, the mirror of per-environment accumulators) and the device (wind_state_kernel).
// Plain C++ apart from the qualifiers, so that a host compiler can build it alone.
#pragma once
#include <math.h>

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
