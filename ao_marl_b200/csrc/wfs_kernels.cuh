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
