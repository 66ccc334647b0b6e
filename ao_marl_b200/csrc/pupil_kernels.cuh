// Per-pixel kernels over the pupil-plane phase: the materialised phase (wfs.get_wfs_phase), the target's phase moments
// and Strehl, geometric slopes, and the centre of gravity of a supplied detector cube.  The phase at a pupil pixel is
// written once, as the screens' part (pupil_screens) and the mirrors' part (pupil_mirrors); the sensor frame kernels
// and the pupil sweep (pupil_sweep.cuh) restate the same arithmetic in their own layouts.
#pragma once
#include <cuda_runtime.h>
#include "rng.cuh"
#include "wfs_params.cuh"

// Atmosphere part of the phase (microns) of pixel (x, y) of the mpupil frame for environment e: bilinear sample of every
// layer, in layer order.  PE: per-environment winds (the layer offsets come from p.wind).  The footprint lies inside the
// screen (checked on the host) and 0 <= ox, oy < N: one conditional subtract wraps.
template <bool PE>
__device__ __forceinline__ float pupil_screens(const WfsParams& p, int e, int x, int y) {
  float acc = 0.f;
  for (int l = 0; l < p.n_layers; ++l) {
    const WfsLayer& L = p.layer[l];
    const int N = L.N;
    const float* scr = L.screen + (size_t)e * N * N;
    const int ox = L.ox[e], oy = L.oy[e];
    const WindRec w = wind_of<PE>(p, l, e);
    int pc0 = x + w.ix + ox; pc0 -= (pc0 >= N) ? N : 0;
    int pc1 = pc0 + 1;       pc1 -= (pc1 >= N) ? N : 0;
    int pr0 = y + w.iy + oy; pr0 -= (pr0 >= N) ? N : 0;
    int pr1 = pr0 + 1;       pr1 -= (pr1 >= N) ? N : 0;
    float top = wfs_layer_row(scr, N, pr0, pc0, pc1, w.fx);
    float bot = wfs_layer_row(scr, N, pr1, pc0, pc1, w.fx);
    acc += top + w.fy * (bot - top);
  }
  return acc;
}

// Mirror part of the phase of pixel (x, y) for environment e: stamp superposition evaluated through the lattice
// directly, then the two tip-tilt planes.
__device__ __forceinline__ float pupil_mirrors(const WfsParams& p, int e, int x, int y) {
  const float* volts = p.volts + (size_t)e * p.ldv;
  const int X = x + p.pzt_off, Y = y + p.pzt_off;
  float dm = 0.f;
  int gxh = (X - p.i1_0) >= 0 ? (X - p.i1_0) / p.pitch : -1;
  int gyh = (Y - p.j1_0) >= 0 ? (Y - p.j1_0) / p.pitch : -1;
  for (int gy = gyh; gy >= 0 && Y - (p.j1_0 + gy * p.pitch) < p.ss; --gy) {
    if (gy >= p.grid_n) continue;
    float fy = p.stamp1d[Y - (p.j1_0 + gy * p.pitch)];
    for (int gx = gxh; gx >= 0 && X - (p.i1_0 + gx * p.pitch) < p.ss; --gx) {
      if (gx >= p.grid_n) continue;
      int a = p.act_map[gy * p.grid_n + gx];
      if (a >= 0) dm = fmaf(volts[a] * fy, p.stamp1d[X - (p.i1_0 + gx * p.pitch)], dm);
    }
  }
  size_t to = (size_t)(y + p.tt_off) * p.tt_dim + (x + p.tt_off);
  dm = fmaf(volts[p.pzt_nact], p.tt_planes[to], dm);
  dm = fmaf(volts[p.pzt_nact + 1], p.tt_planes[(size_t)p.tt_dim * p.tt_dim + to], dm);
  return dm;
}

// Materialised pupil phase (wfs.get_wfs_phase): one thread per pixel.
template <bool PE = false>
__global__ void wfs_phase_kernel(WfsParams p, float* phase) {
  const int e = blockIdx.z;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= p.n || y >= p.n) return;
  float acc = pupil_screens<PE>(p, e, x, y);
  if (p.use_dm) acc += pupil_mirrors(p, e, x, y);
  phase[((size_t)e * p.n + y) * p.n + x] = acc;
}

// Phase statistics over the pupil for the target's Strehl (TargetCompass.comp_strehl / get_strehl,
// targetCompass.py:139-196: get_strehl()[2] is the phase variance, [0] the peak of the PSF): the phase of
// wfs_phase_kernel is evaluated per pixel and reduced on the fly -- sum m, sum m phi, sum m phi^2, sum m cos(k phi),
// sum m sin(k phi) per environment (double atomics) -- instead of materialising [E][n][n].
// grid (ceil(n/32), ceil(n/8), E), block (32, 8).  (Per-pixel cross-check form of pupil_sweep.cuh MODE 1.)
#define TAR_ACC 12   // floats per environment of the long-exposure accumulators: SE sum, variance sum, 9 core pixels
template <bool PE = false>
__global__ void target_moments_kernel(WfsParams p, double* mom, float k2t, int stride, float core_step) {
  const int e = blockIdx.z;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  float m = 0.f, acc = 0.f;
  if (x < p.n && y < p.n) m = p.mpupil[(size_t)y * p.n + x];
  if (m != 0.f) {
    acc = pupil_screens<PE>(p, e, x, y);
    if (p.use_dm) acc += pupil_mirrors(p, e, x, y);
  }
  // sv[0..4]: m, m phi, m phi^2, m cos, m sin ; with the PSF core (stride > 5, same slots as pupil_sweep.cuh MODE 2):
  // sv[5 + 4 a + j] = T1..T4 of a = -1, 0, +1 ; sv[17..20] = (Re, Im) of (a, b) = (-1, 0), (+1, 0)
  float sv[21];
#pragma unroll
  for (int j = 0; j < 21; ++j) sv[j] = 0.f;
  sv[0] = m; sv[1] = m * acc; sv[2] = m * acc * acc;
  const int nsum = stride > 5 ? 21 : 5;
  if (m != 0.f) {
    float sn, cs;
    sincosf(k2t * acc, &sn, &cs);
    sv[3] = cs * m; sv[4] = sn * m;
    if (stride > 5) {
      float sx, cx, sy, cy;
      sincospif(2.f * (float)x * core_step, &sx, &cx);
      sincospif(2.f * (float)y * core_step, &sy, &cy);
      const float re[3] = {cs * cx - sn * sx, cs, cs * cx + sn * sx}, im[3] = {sn * cx + cs * sx, sn, sn * cx - cs * sx};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        sv[5 + 4 * a] = re[a] * cy; sv[6 + 4 * a] = im[a] * sy; sv[7 + 4 * a] = im[a] * cy; sv[8 + 4 * a] = re[a] * sy;
      }
      sv[17] = re[0]; sv[18] = im[0]; sv[19] = re[2]; sv[20] = im[2];
    }
  }
  __shared__ float red[8][21];
  for (int j = 0; j < nsum; ++j) {
    float t = sv[j];
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) t += __shfl_xor_sync(0xffffffffu, t, sft);
    if (threadIdx.x == 0) red[threadIdx.y][j] = t;
  }
  __syncthreads();
  if (threadIdx.y == 0 && threadIdx.x < nsum) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    if (t != 0.f) atomicAdd(mom + (size_t)e * stride + threadIdx.x, (double)t);
  }
}

// [E][4] = {short-exposure Strehl, long-exposure mean of it, phase variance, running mean variance}.  The short-exposure
// figure is the on-axis intensity ratio |<exp(i k phi)>|^2 over the pupil -- the peak of the PSF of a tilt-free
// residual, what the reference reads off its FFT image; it equals the Marechal value exp(-var k^2) for small residuals
// and stays meaningful in open loop where that underflows.  The long-exposure PSF is the mean of the short ones, so
// its peak is the running mean.  acc [E][2] running sums of SE and var, n_le the number of accumulated frames
// including this one (0: no accumulation).
// le_n [E] (or null): per-environment counts once environments are staggered (aom_reset_envs), advanced here when n_le > 0;
// an environment whose first step is pending (first[e]) is left untouched.
__global__ void target_strehl_kernel(const double* mom, int stride, float* strehl, float* acc, int E, int n_le, int* le_n,
                                     const int* first) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  if (le_n) {
    if (first[e]) return;
    n_le = n_le > 0 ? ++le_n[e] : 0;
  }
  const double* m = mom + (size_t)e * stride;
  const double s0 = m[0], s1 = m[1], s2 = m[2], sc = m[3], ss = m[4];
  float var = 0.f, se = 1.f;
  if (s0 > 0.0) {
    const double mean = s1 / s0;
    var = (float)fmax(s2 / s0 - mean * mean, 0.0);
    se = (float)((sc * sc + ss * ss) / (s0 * s0));
  }
  strehl[e * 4 + 0] = se;
  strehl[e * 4 + 2] = var;
  if (n_le > 0) {
    acc[e * TAR_ACC + 0] += se;
    acc[e * TAR_ACC + 1] += var;
    strehl[e * 4 + 1] = acc[e * TAR_ACC + 0] / (float)n_le;
    strehl[e * 4 + 3] = acc[e * TAR_ACC + 1] / (float)n_le;
  }
}

// Geometric slopes of a materialised pupil phase [E][n][n] (RtcCompass.do_centroids_geom, rtcCompass.py; sutra slopes_geom,
// un-vendored -- the convention of oracle/aoframe.py::slopes_geom and init/rtc.py::geometric_slopes, which the actuator
// filtering of the reference's imat_geom pins): central differences inside the 16 x 16 tile, one-sided at its edge, masked
// by the pupil, summed / pdiam / 2, times alpha = 0.206265 / subaperture size, divided by the subaperture's flux fraction.
// grid (nvalid, E), block 256 (one thread per pixel of the tile).
__global__ void __launch_bounds__(256) slopes_geom_kernel(WfsParams p, const float* __restrict__ phase, float* __restrict__ slopes,
                                                          int lds, float alpha) {
  const int k = blockIdx.x, e = blockIdx.y;
  const int r = threadIdx.x >> 4, c = threadIdx.x & 15;
  const int x0 = p.sub_x0[k], y0 = p.sub_y0[k];
  const float* ph = phase + (size_t)e * p.n * p.n;
  auto at = [&](int rr, int cc) { return ph[(size_t)(y0 + rr) * p.n + x0 + cc]; };
  const float m = p.mpupil[(size_t)(y0 + r) * p.n + x0 + c];
  const float gx = (c == 0) ? at(r, 1) - at(r, 0) : (c == 15) ? at(r, 15) - at(r, 14) : at(r, c + 1) - at(r, c - 1);
  const float gy = (r == 0) ? at(1, c) - at(0, c) : (r == 15) ? at(15, c) - at(14, c) : at(r + 1, c) - at(r - 1, c);
  float sx = gx * m, sy = gy * m;
#pragma unroll
  for (int sft = 16; sft > 0; sft >>= 1) {
    sx += __shfl_xor_sync(0xffffffffu, sx, sft);
    sy += __shfl_xor_sync(0xffffffffu, sy, sft);
  }
  __shared__ float red[2][8];
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sx; red[1][threadIdx.x >> 5] = sy; }
  __syncthreads();
  if (threadIdx.x < 2) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
    slopes[(size_t)e * lds + threadIdx.x * p.nvalid + k] = t / 16.f / 2.f * alpha / p.flux[k];
  }
}

// Centre of gravity of an externally supplied detector cube [E][nvalid][256] (denoiser path).
__global__ void cog_kernel(const float* cube, float* slopes, int lds, int nvalid, long long total,
                           float cog_offset, float pixsize) {
  const int lane = threadIdx.x & 31;
  long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= total) return;
  const int e = (int)(w / nvalid), k = (int)(w % nvalid);
  const float* c = cube + (size_t)w * 256;
  float s0 = 0.f, sy = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = c[lane + 32 * j];
    s0 += v;
    sy += v * (float)((lane + 32 * j) >> 4);
  }
  float sx = s0 * (float)(lane & 15);
#pragma unroll
  for (int sft = 16; sft > 0; sft >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
    sx += __shfl_xor_sync(0xffffffffu, sx, sft);
    sy += __shfl_xor_sync(0xffffffffu, sy, sft);
  }
  if (lane == 0) {
    float gx = (s0 > 0.f) ? sx / s0 : cog_offset;
    float gy = (s0 > 0.f) ? sy / s0 : cog_offset;
    slopes[(size_t)e * lds + k] = (gx - cog_offset) * pixsize;
    slopes[(size_t)e * lds + nvalid + k] = (gy - cog_offset) * pixsize;
  }
}

// Photon and read noise of n detector pixels of mean lam (aom_pixel_noise): the sensor kernels' draw, one counter per pixel
__global__ void pixel_noise_kernel(const float* lam, float* out, long long n, float noise, uint32_t k0,
                                   uint32_t k1, uint32_t frame, uint32_t wfs) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = aom_pixel_noise(lam[i], noise, (uint32_t)i, frame, wfs, k0, k1);
}
