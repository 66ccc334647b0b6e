// Shack-Hartmann frame, fused: raytrace through the layers -> + mirror surfaces -> complex pupil
// field -> pruned 2-D DFT in shared memory -> |.|^2 -> nrebin x nrebin binning -> flux
// normalisation -> photon / read noise -> centre of gravity.   One warp owns one subaperture of one
// environment; nothing but the slopes (and, on request, the 16 x 16 spot) goes back to HBM.
//
// Replaces, per frame, sutra's raytrace + fillcamplipup + batched cuFFT + abs2 + fillbincube +
// noise + centroid kernels behind WfsCompass.raytrace / compute_wfs_image / RtcCompass.do_centroids
// (shesha/supervisor/components/wfsCompass.py:334-343, sourceCompass.py:54-85, rtcCompass.py:557-563);
// the algorithm is the one the reference's tables define (shesha/init/geom_init.py:622-811) and
// oracle/aoframe.py restates.
#pragma once
#include <cuda_runtime.h>
#include "fft16.cuh"
#include "wfs_params.cuh"

#define WFS_WARPS 8
#define WFS_PD 16
#define WFS_NPIX 16
#define WFS_IN_STRIDE 18
#define WFS_NG_MAX 6

// phase (microns) of pixel (y, x) of the mpupil frame for environment e: atmosphere part
__device__ __forceinline__ float wfs_layer_row(const float* scr, int N, int prow, int pc0, int pc1, float fx) {
  const float* r = scr + (size_t)prow * N;
  float a = __ldg(r + pc0), b = __ldg(r + pc1);
  return a + fx * (b - a);
}

// PE: per-environment winds (the layer offsets come from p.wind)
// NE: per-environment sensor values (each environment's noise and photon count from p.noise_env / p.nph_env)
template <int R, bool PE = false, bool NE = false>
__global__ void __launch_bounds__(WFS_WARPS * 32, 2) wfs_frame_kernel(WfsParams p) {
  constexpr int NFFT = 16 * R;
  constexpr int H = 4 * R;            // half width of the kept spectrum
  constexpr int W = 2 * H;            // kept spectrum width = npix * nrebin
  constexpr int NREBIN = W / WFS_NPIX;
  constexpr int XS = W + R;           // row stride of the intermediate (bank-conflict free)
  constexpr int WARP_FLOATS = 2 * 16 * WFS_IN_STRIDE + 2 * 16 * XS + 256 + 40 + WFS_NG_MAX * 16;

  extern __shared__ __align__(16) float smem[];
  float* s_twr = smem;                       // [R][16]
  float* s_twi = s_twr + R * 16;
  float* s_f = s_twi + R * 16;               // [64] separable stamp factor
  float* s_half = s_f + 64;                  // [256]
  float* warp_base = s_half + 256;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_inr = warp_base + warp * WARP_FLOATS;   // [16][18]
  float* s_ini = s_inr + 16 * WFS_IN_STRIDE;
  float* s_x1r = s_ini + 16 * WFS_IN_STRIDE;       // [16][XS]
  float* s_x1i = s_x1r + 16 * XS;
  float* s_img = s_x1i + 16 * XS;                  // [16][16]
  float* s_v = s_img + 256;                        // [<=36] actuator volts of the neighbourhood (+2 tt)
  float* s_t = s_v + 40;                           // [NG][16]

  for (int i = threadIdx.x; i < R * 16; i += blockDim.x) {
    int b = i / 16, nn = i % 16;
    float sn, cs;
    sincospif(-2.0f * (float)(b * nn) / (float)NFFT, &sn, &cs);
    s_twr[i] = cs;
    s_twi[i] = sn;
  }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_f[i] = (i < p.ss) ? p.stamp1d[i] : 0.f;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_half[i] = p.halfxy[i];
  __syncthreads();

  const long long total = (long long)p.E * p.nvalid;
  const int hx = lane & 15;            // pixel column owned in the load phase
  const int hy = (lane >> 4) * 8;      // first of the 8 rows owned
  for (long long w = (long long)blockIdx.x * WFS_WARPS + warp; w < total; w += (long long)gridDim.x * WFS_WARPS) {
    const int e = (int)(w / p.nvalid);
    const int k = (int)(w % p.nvalid);
    const int x0 = p.sub_x0[k], y0 = p.sub_y0[k];
    float ph[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) ph[i] = 0.f;

    // ---- atmosphere: bilinear sample of every layer (ring-buffered screens) ----
    for (int l = 0; l < p.n_layers; ++l) {
      const WfsLayer& L = p.layer[l];
      const int N = L.N;
      const float* scr = L.screen + (size_t)e * N * N;
      const int ox = L.ox[e], oy = L.oy[e];
      const WindRec w = wind_of<PE>(p, l, e);
      int pc0 = x0 + hx + w.ix + ox;  pc0 -= (pc0 >= N) ? N : 0;  pc0 -= (pc0 >= N) ? N : 0;
      int pc1 = pc0 + 1;              pc1 -= (pc1 >= N) ? N : 0;
      int pr = y0 + hy + w.iy + oy;   pr -= (pr >= N) ? N : 0;    pr -= (pr >= N) ? N : 0;
      float prev = wfs_layer_row(scr, N, pr, pc0, pc1, w.fx);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        pr += 1; pr -= (pr >= N) ? N : 0;
        float cur = wfs_layer_row(scr, N, pr, pc0, pc1, w.fx);
        ph[i] += prev + w.fy * (cur - prev);
        prev = cur;
      }
    }

    // ---- mirrors: separable stamp superposition + two tip-tilt planes ----
    if (p.use_dm) {
      const float* volts = p.volts + (size_t)e * p.ldv;
      const int X0 = x0 + p.pzt_off, Y0 = y0 + p.pzt_off;       // tile origin in the DM support
      // lattice columns / rows whose stamp [i1, i1+ss) meets [X0, X0+16)
      const int dxm = X0 - p.i1_0 - (p.ss - 1);
      const int gx_lo = (dxm >= 0) ? (dxm + p.pitch - 1) / p.pitch : -((-dxm) / p.pitch);
      const int dym = Y0 - p.j1_0 - (p.ss - 1);
      const int gy_lo = (dym >= 0) ? (dym + p.pitch - 1) / p.pitch : -((-dym) / p.pitch);
      for (int c = lane; c < WFS_NG_MAX * WFS_NG_MAX; c += 32) {
        int gy = gy_lo + c / WFS_NG_MAX, gx = gx_lo + c % WFS_NG_MAX;
        float v = 0.f;
        if (gx >= 0 && gx < p.grid_n && gy >= 0 && gy < p.grid_n) {
          int a = p.act_map[gy * p.grid_n + gx];
          if (a >= 0) v = volts[a];
        }
        s_v[c] = v;
      }
      if (lane < 2) s_v[36 + lane] = volts[p.pzt_nact + lane];
      __syncwarp();
      // T[g][x] = sum_gx V[g][gx] f[x + X0 - i1(gx)]
      for (int t = lane; t < WFS_NG_MAX * 16; t += 32) {
        int g = t >> 4, x = t & 15;
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < WFS_NG_MAX; ++j) {
          int a = X0 + x - (p.i1_0 + (gx_lo + j) * p.pitch);
          float fv = (a >= 0 && a < p.ss) ? s_f[a] : 0.f;
          acc = fmaf(s_v[g * WFS_NG_MAX + j], fv, acc);
        }
        s_t[t] = acc;
      }
      __syncwarp();
      const float tt0 = s_v[36], tt1 = s_v[37];
      const float* plane0 = p.tt_planes;
      const float* plane1 = p.tt_planes + (size_t)p.tt_dim * p.tt_dim;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int y = hy + i;
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < WFS_NG_MAX; ++j) {
          int b = Y0 + y - (p.j1_0 + (gy_lo + j) * p.pitch);
          float fv = (b >= 0 && b < p.ss) ? s_f[b] : 0.f;
          acc = fmaf(fv, s_t[j * 16 + hx], acc);
        }
        size_t to = (size_t)(y0 + y + p.tt_off) * p.tt_dim + (x0 + hx + p.tt_off);
        acc = fmaf(tt0, __ldg(plane0 + to), acc);
        acc = fmaf(tt1, __ldg(plane1 + to), acc);
        ph[i] += acc;
      }
    }

    // ---- complex field of the subaperture ----
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int y = hy + i;
      const float m = __ldg(p.mpupil + (size_t)(y0 + y) * p.n + x0 + hx);
      const float arg = p.k2 * ph[i] - s_half[y * 16 + hx];
      float sn, cs;
      sincosf(arg, &sn, &cs);
      s_inr[y * WFS_IN_STRIDE + hx] = m * cs;
      s_ini[y * WFS_IN_STRIDE + hx] = m * sn;
    }
    __syncwarp();

    // ---- row pass: 16 rows x R phase classes ----
    {
      float outr[8], outi[8];
#pragma unroll 1
      for (int it = 0; it < (16 * R) / 32; ++it) {
        const int task = it * 32 + lane;
        const int row = task / R, b = task % R;
        aom_fft16_pruned(s_inr + row * WFS_IN_STRIDE, s_ini + row * WFS_IN_STRIDE, s_twr + b * 16,
                         s_twi + b * 16, outr, outi);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          s_x1r[row * XS + H + R * q + b] = outr[q];
          s_x1i[row * XS + H + R * q + b] = outi[q];
          s_x1r[row * XS + R * q + b] = outr[4 + q];
          s_x1i[row * XS + R * q + b] = outi[4 + q];
        }
      }
    }
    __syncwarp();

    // ---- column pass + |.|^2 + binning ----
    {
      float vr[16], vi[16], outr[8], outi[8];
#pragma unroll 1
      for (int it = 0; it < (W * R) / 32; ++it) {
        const int task = it * 32 + lane;
        const int c = task / R, b = task % R;
#pragma unroll
        for (int nn = 0; nn < 16; ++nn) {
          vr[nn] = s_x1r[nn * XS + c];
          vi[nn] = s_x1i[nn * XS + c];
        }
        aom_fft16_pruned(vr, vi, s_twr + b * 16, s_twi + b * 16, outr, outi);
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          float v = outr[o] * outr[o] + outi[o] * outi[o];
#pragma unroll
          for (int sft = 1; sft < NREBIN; sft <<= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);       // over b
#pragma unroll
          for (int sft = R; sft < R * NREBIN; sft <<= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);   // over c
          if ((b % NREBIN) == 0 && (c % NREBIN) == 0) {
            const int q = o & 3;
            const int ky = ((o < 4) ? H : 0) + R * q + b;       // centred row of the spectrum
            s_img[(ky / NREBIN) * 16 + c / NREBIN] = v;
          }
        }
      }
    }
    __syncwarp();

    // ---- flux normalisation, noise, centre of gravity ----
    float px[8];
    float tot = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { px[j] = s_img[lane + 32 * j]; tot += px[j]; }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, sft);
    const float scale = nphotons_of<NE>(p, e) * p.flux[k] / tot;
    const float noise = noise_of<NE>(p, e);
    const uint32_t k0 = p.k0[e], k1 = p.k1[e], fr = noise_frame(p, e);
    float s0 = 0.f, sy = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int pidx = lane + 32 * j;
      float v = px[j] * scale;
      v = aom_pixel_noise(v, noise, (uint32_t)(k * 256 + pidx), fr, p.wfs_index, k0, k1);
      px[j] = v;
      s0 += v;
      sy += v * (float)(pidx >> 4);
    }
    float sx = s0 * (float)(lane & 15);
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
      sx += __shfl_xor_sync(0xffffffffu, sx, sft);
      sy += __shfl_xor_sync(0xffffffffu, sy, sft);
    }
    if (p.bincube) {
      float* out = p.bincube + ((size_t)e * p.nvalid + k) * 256;
#pragma unroll
      for (int j = 0; j < 8; ++j) out[lane + 32 * j] = px[j];
    }
    if (lane == 0) {
      float gx = (s0 > 0.f) ? sx / s0 : p.cog_offset;
      float gy = (s0 > 0.f) ? sy / s0 : p.cog_offset;
      float* sl = p.slopes + (size_t)e * p.lds;
      sl[k] = (gx - p.cog_offset) * p.pixsize;
      sl[p.nvalid + k] = (gy - p.cog_offset) * p.pixsize;
    }
    __syncwarp();
  }
}

template <int R>
constexpr size_t wfs_smem_bytes() {
  return sizeof(float) * (size_t)(2 * R * 16 + 64 + 256 +
                                  WFS_WARPS * (2 * 16 * WFS_IN_STRIDE + 2 * 16 * (8 * R + R) + 256 + 40 + WFS_NG_MAX * 16));
}

// Materialised pupil phase (wfs.get_wfs_phase): one thread per pixel, same arithmetic as above but
// with the mirror surface evaluated through the lattice directly.
template <bool PE = false>
__global__ void wfs_phase_kernel(WfsParams p, float* phase) {
  const int e = blockIdx.z;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= p.n || y >= p.n) return;
  float acc = 0.f;
  for (int l = 0; l < p.n_layers; ++l) {
    const WfsLayer& L = p.layer[l];
    const int N = L.N;
    const float* scr = L.screen + (size_t)e * N * N;
    const int ox = L.ox[e], oy = L.oy[e];
    const WindRec w = wind_of<PE>(p, l, e);
    int pc0 = (x + w.ix + ox) % N, pc1 = (pc0 + 1) % N;
    int pr0 = (y + w.iy + oy) % N, pr1 = (pr0 + 1) % N;
    float top = wfs_layer_row(scr, N, pr0, pc0, pc1, w.fx);
    float bot = wfs_layer_row(scr, N, pr1, pc0, pc1, w.fx);
    acc += top + w.fy * (bot - top);
  }
  if (p.use_dm) {
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
    acc += dm;
  }
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
    for (int l = 0; l < p.n_layers; ++l) {
      const WfsLayer& L = p.layer[l];
      const int N = L.N;
      const float* scr = L.screen + (size_t)e * N * N;
      const int ox = L.ox[e], oy = L.oy[e];
      const WindRec w = wind_of<PE>(p, l, e);
      int pc0 = (x + w.ix + ox) % N, pc1 = (pc0 + 1) % N;
      int pr0 = (y + w.iy + oy) % N, pr1 = (pr0 + 1) % N;
      float top = wfs_layer_row(scr, N, pr0, pc0, pc1, w.fx);
      float bot = wfs_layer_row(scr, N, pr1, pc0, pc1, w.fx);
      acc += top + w.fy * (bot - top);
    }
    if (p.use_dm) {
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
      acc += dm;
    }
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
