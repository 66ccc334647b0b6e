// Shack-Hartmann frame on the tensor pipe (Nfft = 64, nrebin = 2 geometry of the production files).
//
// Same fused pipeline as wfs_frame_kernel (raytrace -> mirrors -> complex field -> pruned 2-D DFT ->
// |.|^2 -> 2 x 2 binning -> flux normalisation -> noise -> centre of gravity, one warp per subaperture)
// but the DFT is two chained real GEMMs issued as warp-level m16n8k16 tensor-core MMAs whose operands
// never leave the register file:
//
//   stage 1   [Tr;Ti] (64 x 16) = [[Wr,-Wi],[Wi,Wr]] (64 x 32) . [Xr;Xi]^T (32 x 16)     contraction over x
//   stage 2   [Yr|Yi] (32 x 64) = [Tr|Ti] (32 x 32) . [[Wr,Wi],[-Wi,Wr]] (32 x 64)       contraction over y
//
// W[n][i] = exp(-2 pi i n F(i) / 64) with F the 32 kept frequencies (0..15, 48..63: the only bins the
// reference's binmap reads, geom_init.py:731-758).  The accumulator fragment of stage 1 has exactly the
// register layout of the A fragment of stage 2, so T goes from one MMA to the next through a
// float -> half2 conversion only.  fp32 accuracy comes from an error-free split of every operand into
// two halves (x = hi + lo, 11 + 11 significant bits) and three MMAs per product (hi.hi + hi.lo + lo.hi);
// the dropped lo.lo term is 2^-22 relative.  Slopes then agree with a float32 FFT to ~1e-7 relative.
//
// Replaces sutra's fillcamplipup + batched cuFFT + abs2 + fillbincube + centroid kernels behind
// WfsCompass.compute_wfs_image / RtcCompass.do_centroids (wfsCompass.py:334-343, rtcCompass.py:557-563).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include "device_common.cuh"
#include "wfs_kernels.cuh"

#define WFM_WARPS 8
#define WFM_WARP_FLOATS (40 + 2 * WFS_NG_MAX * 16)

__device__ __forceinline__ void wfm_mma(float (&c)[4], const uint4& a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t wfm_pack(float lo_elem, float hi_elem) {
  __half2 h = __floats2half2_rn(lo_elem, hi_elem);
  return *reinterpret_cast<uint32_t*>(&h);
}

// error-free split of a pair: hi keeps the leading 11 significant bits (exactly representable in
// fp16 over the value range of the fields, |v| <= 16), lo the remainder
__device__ __forceinline__ void wfm_split(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
  const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  hi = wfm_pack(ah, bh);
  lo = wfm_pack(a - ah, b - bh);
}

// rounded split for the constant twiddles
__device__ __forceinline__ void wfm_split_rn(float v, float& hi, float& lo) {
  hi = __half2float(__float2half_rn(v));
  lo = v - hi;
}

// W[n][i], i = index in the kept-frequency list
__device__ __forceinline__ float wfm_w(int n, int i, int part) {
  const int F = (i < 16) ? i : i + 32;
  const int ang = (n * F) & 63;
  float s, c;
  sincospif(-(float)ang * (1.0f / 32.0f), &s, &c);
  return part ? s : c;
}

// three consecutive floats p[0..2]; `even` = p is 8-byte aligned (warp-uniform), else p + 1 is
__device__ __forceinline__ void wfm_load3(const float* __restrict__ p, bool even, float& v0, float& v1, float& v2) {
  if (even) {
    const float2 a = __ldg(reinterpret_cast<const float2*>(p));
    v0 = a.x; v1 = a.y; v2 = __ldg(p + 2);
  } else {
    const float2 b = __ldg(reinterpret_cast<const float2*>(p + 1));
    v0 = __ldg(p); v1 = b.x; v2 = b.y;
  }
}

// bilinear sample of one layer at the 8 pixels of this lane: tile rows 4 rg .. 4 rg + 3, cols 2 xp, 2 xp + 1.
// Fast path (tile does not meet the ring seam): five rows of three consecutive floats, 64-bit loads.
__device__ __forceinline__ void wfm_layer(const float* __restrict__ scr, int N, int tr0, int tc0, int rg, int xp,
                                          float fx, float fy, float (&ph)[4][2]) {
  float h[5][2];
  if (tc0 + 16 < N && tr0 + 16 < N && !(N & 1)) {
    const float* base = scr + (size_t)(tr0 + 4 * rg) * N + tc0 + 2 * xp;
    const bool even = !(tc0 & 1);
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      float v0, v1, v2;
      wfm_load3(base + (size_t)r * N, even, v0, v1, v2);
      h[r][0] = v0 + fx * (v1 - v0);
      h[r][1] = v1 + fx * (v2 - v1);
    }
  } else {
    int cc[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { cc[i] = tc0 + 2 * xp + i; cc[i] -= (cc[i] >= N) ? N : 0; }
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      int rr = tr0 + 4 * rg + r;
      rr -= (rr >= N) ? N : 0;
      const float* rp = scr + (size_t)rr * N;
      const float v0 = __ldg(rp + cc[0]), v1 = __ldg(rp + cc[1]), v2 = __ldg(rp + cc[2]);
      h[r][0] = v0 + fx * (v1 - v0);
      h[r][1] = v1 + fx * (v2 - v1);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    ph[i][0] += h[i][0] + fy * (h[i + 1][0] - h[i][0]);
    ph[i][1] += h[i][1] + fy * (h[i + 1][1] - h[i][1]);
  }
}

// PASS2_FULL = 1: three MMAs per product in both stages (fp32-grade).  0 drops the W-lo pass of stage 2.
// NL: number of turbulence layers traced (compile-time so that the layer loop unrolls and its loads overlap),
//     -1 = run-time count.
template <int PASS2_FULL, int NL>
__global__ void __launch_bounds__(WFM_WARPS * 32, 2) wfs_frame_mma_kernel(WfsParams p) {
  __shared__ uint4 s_c1[8][32];     // stage-1 A fragments: [mt*4 + part*2 + hl][lane]
  __shared__ uint4 s_c2[8][32];     // stage-2 B fragments: [b*2 + hl][lane] = {Wr b0, Wr b1, Wi b0, Wi b1}
  __shared__ float s_f[64];         // separable stamp factor
  __shared__ __align__(16) float s_half[256];
  __shared__ __align__(16) float s_warp[WFM_WARPS][WFM_WARP_FLOATS];
  __shared__ uint4 s_frag[WFM_WARPS][4][32];   // field fragments in flight: [part*2 + hl][lane] = {j0h0, j0h1, j1h0, j1h1}

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, q = lane & 3;       // MMA fragment coordinates
  const int xp = lane & 7, rg = lane >> 3;     // load-phase pixels: rows 4 rg .. 4 rg + 3, cols 2 xp, 2 xp + 1

  for (int t = threadIdx.x; t < 16 * 32; t += blockDim.x) {
    const int c = t >> 5, l = t & 31, lg = l >> 2, lq = l & 3;
    float v[8];
    const int hl = c & 1;
    if (c < 8) {
      const int mt = c >> 2, part = (c >> 1) & 1;
      const int rows[2] = {lg, lg + 8};
      const int cols[4] = {2 * lq, 2 * lq + 1, 2 * lq + 8, 2 * lq + 9};
      // a0 = (g; 2q, 2q+1)  a1 = (g+8; 2q, 2q+1)  a2 = (g; 2q+8, 2q+9)  a3 = (g+8; 2q+8, 2q+9)
#pragma unroll
      for (int reg = 0; reg < 4; ++reg)
#pragma unroll
        for (int e = 0; e < 2; ++e) v[reg * 2 + e] = wfm_w(cols[(reg >> 1) * 2 + e], 16 * mt + rows[reg & 1], part);
    } else {
      const int b = (c - 8) >> 1;
      const int ks[4] = {2 * lq, 2 * lq + 1, 2 * lq + 8, 2 * lq + 9};
      // {Wr b0, Wr b1, Wi b0, Wi b1}, b0 = (k = 2q, 2q+1; n = g), b1 = (k = 2q+8, 2q+9; n = g)
#pragma unroll
      for (int reg = 0; reg < 4; ++reg)
#pragma unroll
        for (int e = 0; e < 2; ++e) v[reg * 2 + e] = wfm_w(ks[(reg & 1) * 2 + e], 8 * b + lg, reg >> 1);
    }
    uint32_t w[4];
#pragma unroll
    for (int reg = 0; reg < 4; ++reg) {
      float h0, l0, h1, l1;
      wfm_split_rn(v[reg * 2], h0, l0);
      wfm_split_rn(v[reg * 2 + 1], h1, l1);
      w[reg] = hl ? wfm_pack(l0, l1) : wfm_pack(h0, h1);
    }
    uint4 o = make_uint4(w[0], w[1], w[2], w[3]);
    if (c < 8) s_c1[c][l] = o; else s_c2[c - 8][l] = o;
  }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_f[i] = (p.use_dm && i < p.ss) ? p.stamp1d[i] : 0.f;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_half[i] = p.halfxy[i];
  __syncthreads();

  float* s_v = s_warp[warp];                 // [<=36] actuator volts of the neighbourhood (+2 tt)
  float* s_t = s_v + 40;                     // [NG][16]  T[j][x]  = sum_gx V[j][gx] f[x + X0 - i1(gx)]
  float* s_fy = s_t + WFS_NG_MAX * 16;       // [NG][16]  FY[j][y] = f[y + Y0 - j1(gy_lo + j)]
  uint32_t* s_fw = reinterpret_cast<uint32_t*>(&s_frag[warp][0][0]);
  const int n_layers = (NL >= 0) ? NL : p.n_layers;

  const long long total = (long long)p.E * p.nvalid;
  for (long long w = (long long)blockIdx.x * WFM_WARPS + warp; w < total; w += (long long)gridDim.x * WFM_WARPS) {
    const int e = (int)(w / p.nvalid);
    const int k = (int)(w % p.nvalid);
    const int x0 = p.sub_x0[k], y0 = p.sub_y0[k];
    float ph[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) ph[i][0] = ph[i][1] = 0.f;

    // ---- atmosphere ----
#pragma unroll
    for (int l = 0; l < n_layers; ++l) {
      const WfsLayer& L = p.layer[l];
      const int N = L.N;
      const float* scr = L.screen + (size_t)e * N * N;
      int tc0 = x0 + L.ix + L.ox[e];  tc0 -= (tc0 >= N) ? N : 0;  tc0 -= (tc0 >= N) ? N : 0;
      int tr0 = y0 + L.iy + L.oy[e];  tr0 -= (tr0 >= N) ? N : 0;  tr0 -= (tr0 >= N) ? N : 0;
      wfm_layer(scr, N, tr0, tc0, rg, xp, L.fx, L.fy, ph);
    }

    // ---- mirrors: separable stamp superposition + two tip-tilt planes ----
    if (p.use_dm) {
      const float* volts = p.volts + (size_t)e * p.ldv;
      const int X0 = x0 + p.pzt_off, Y0 = y0 + p.pzt_off;       // tile origin in the DM support
      const int dxm = X0 - p.i1_0 - (p.ss - 1);
      const int gx_lo = (dxm >= 0) ? (dxm + p.pitch - 1) / p.pitch : -((-dxm) / p.pitch);
      const int dym = Y0 - p.j1_0 - (p.ss - 1);
      const int gy_lo = (dym >= 0) ? (dym + p.pitch - 1) / p.pitch : -((-dym) / p.pitch);
      for (int c = lane; c < WFS_NG_MAX * WFS_NG_MAX; c += 32) {
        const int gy = gy_lo + c / WFS_NG_MAX, gx = gx_lo + c % WFS_NG_MAX;
        float v = 0.f;
        if (gx >= 0 && gx < p.grid_n && gy >= 0 && gy < p.grid_n) {
          const int a = p.act_map[gy * p.grid_n + gx];
          if (a >= 0) v = volts[a];
        }
        s_v[c] = v;
      }
      if (lane < 2) s_v[36 + lane] = volts[p.pzt_nact + lane];
#pragma unroll
      for (int t = lane; t < WFS_NG_MAX * 16; t += 32) {
        const int j = t >> 4, y = t & 15;
        const int b = Y0 + y - (p.j1_0 + (gy_lo + j) * p.pitch);
        s_fy[t] = (b >= 0 && b < p.ss) ? s_f[b] : 0.f;
      }
      __syncwarp();
#pragma unroll
      for (int t = lane; t < WFS_NG_MAX * 16; t += 32) {
        const int j = t >> 4, x = t & 15;
        float acc = 0.f;
#pragma unroll
        for (int jj = 0; jj < WFS_NG_MAX; ++jj) {
          const int a = X0 + x - (p.i1_0 + (gx_lo + jj) * p.pitch);
          const float fv = (a >= 0 && a < p.ss) ? s_f[a] : 0.f;
          acc = fmaf(s_v[j * WFS_NG_MAX + jj], fv, acc);
        }
        s_t[t] = acc;
      }
      __syncwarp();
      const float tt0 = s_v[36], tt1 = s_v[37];
      float acc[4][2];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.f;
#pragma unroll
      for (int j = 0; j < WFS_NG_MAX; ++j) {
        const float2 t2 = *reinterpret_cast<const float2*>(s_t + j * 16 + 2 * xp);
        const float4 f4 = *reinterpret_cast<const float4*>(s_fy + j * 16 + 4 * rg);
        acc[0][0] = fmaf(f4.x, t2.x, acc[0][0]); acc[0][1] = fmaf(f4.x, t2.y, acc[0][1]);
        acc[1][0] = fmaf(f4.y, t2.x, acc[1][0]); acc[1][1] = fmaf(f4.y, t2.y, acc[1][1]);
        acc[2][0] = fmaf(f4.z, t2.x, acc[2][0]); acc[2][1] = fmaf(f4.z, t2.y, acc[2][1]);
        acc[3][0] = fmaf(f4.w, t2.x, acc[3][0]); acc[3][1] = fmaf(f4.w, t2.y, acc[3][1]);
      }
      const float* plane0 = p.tt_planes;
      const float* plane1 = p.tt_planes + (size_t)p.tt_dim * p.tt_dim;
      const bool tt_even = !((x0 + p.tt_off) & 1) && !(p.tt_dim & 1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const size_t to = (size_t)(y0 + 4 * rg + i + p.tt_off) * p.tt_dim + (x0 + 2 * xp + p.tt_off);
        float2 a, b;
        if (tt_even) {
          a = __ldg(reinterpret_cast<const float2*>(plane0 + to));
          b = __ldg(reinterpret_cast<const float2*>(plane1 + to));
        } else {
          a = make_float2(__ldg(plane0 + to), __ldg(plane0 + to + 1));
          b = make_float2(__ldg(plane1 + to), __ldg(plane1 + to + 1));
        }
        ph[i][0] += fmaf(tt1, b.x, fmaf(tt0, a.x, acc[i][0]));
        ph[i][1] += fmaf(tt1, b.y, fmaf(tt0, a.y, acc[i][1]));
      }
    }

    // ---- complex field, split into fp16 hi / lo and transposed through shared memory into B fragments ----
    {
      const bool pup_even = !((x0 | p.n) & 1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int y = 4 * rg + i;
        const float* mp = p.mpupil + (size_t)(y0 + y) * p.n + x0 + 2 * xp;
        const float2 m = pup_even ? __ldg(reinterpret_cast<const float2*>(mp)) : make_float2(__ldg(mp), __ldg(mp + 1));
        const float2 hf = *reinterpret_cast<const float2*>(s_half + y * 16 + 2 * xp);
        float s0, c0, s1, c1;
        wfm_sincos(p.k2 * ph[i][0] - hf.x, s0, c0);
        wfm_sincos(p.k2 * ph[i][1] - hf.y, s1, c1);
        uint32_t rh, rl, ih, il;
        wfm_split(m.x * c0, m.y * c1, rh, rl);
        wfm_split(m.x * s0, m.y * s1, ih, il);
        // fragment word of pixel pair (y; 2xp, 2xp+1): lane' = (y & 7) * 4 + (xp & 3), reg = (y >> 3) * 2 + (xp >> 2)
        const int word = (((y & 7) * 4 + (xp & 3)) << 2) + ((y >> 3) << 1) + (xp >> 2);
        s_fw[0 * 128 + word] = rh;
        s_fw[1 * 128 + word] = rl;
        s_fw[2 * 128 + word] = ih;
        s_fw[3 * 128 + word] = il;
      }
    }
    __syncwarp();
    uint32_t xr_h[2][2], xr_l[2][2], xi_h[2][2], xi_l[2][2];
    {
      const uint4 f0 = s_frag[warp][0][lane], f1 = s_frag[warp][1][lane];
      const uint4 f2 = s_frag[warp][2][lane], f3 = s_frag[warp][3][lane];
      xr_h[0][0] = f0.x; xr_h[0][1] = f0.y; xr_h[1][0] = f0.z; xr_h[1][1] = f0.w;
      xr_l[0][0] = f1.x; xr_l[0][1] = f1.y; xr_l[1][0] = f1.z; xr_l[1][1] = f1.w;
      xi_h[0][0] = f2.x; xi_h[0][1] = f2.y; xi_h[1][0] = f2.z; xi_h[1][1] = f2.w;
      xi_l[0][0] = f3.x; xi_l[0][1] = f3.y; xi_l[1][0] = f3.z; xi_l[1][1] = f3.w;
    }

    // ---- stage 1: T[part][mt][j] (16 x 8 accumulator tiles: rows = kept frequency fx, cols = y) ----
    float T[2][2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const uint4 wr_h = s_c1[mt * 4 + 0][lane], wr_l = s_c1[mt * 4 + 1][lane];
      const uint4 wi_h = s_c1[mt * 4 + 2][lane], wi_l = s_c1[mt * 4 + 3][lane];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        float (&tr)[4] = T[0][mt][j];
        float (&ti)[4] = T[1][mt][j];
#pragma unroll
        for (int c = 0; c < 4; ++c) { tr[c] = 0.f; ti[c] = 0.f; }
        const uint32_t nh0 = xi_h[j][0] ^ 0x80008000u, nh1 = xi_h[j][1] ^ 0x80008000u;
        const uint32_t nl0 = xi_l[j][0] ^ 0x80008000u, nl1 = xi_l[j][1] ^ 0x80008000u;
        // Tr = Wr.Xr - Wi.Xi
        wfm_mma(tr, wr_h, xr_h[j][0], xr_h[j][1]);
        wfm_mma(tr, wr_h, xr_l[j][0], xr_l[j][1]);
        wfm_mma(tr, wr_l, xr_h[j][0], xr_h[j][1]);
        wfm_mma(tr, wi_h, nh0, nh1);
        wfm_mma(tr, wi_h, nl0, nl1);
        wfm_mma(tr, wi_l, nh0, nh1);
        // Ti = Wi.Xr + Wr.Xi
        wfm_mma(ti, wi_h, xr_h[j][0], xr_h[j][1]);
        wfm_mma(ti, wi_h, xr_l[j][0], xr_l[j][1]);
        wfm_mma(ti, wi_l, xr_h[j][0], xr_h[j][1]);
        wfm_mma(ti, wr_h, xi_h[j][0], xi_h[j][1]);
        wfm_mma(ti, wr_h, xi_l[j][0], xi_l[j][1]);
        wfm_mma(ti, wr_l, xi_h[j][0], xi_h[j][1]);
      }
    }

    // ---- stage-2 A fragments: a0 = tile(j=0) c0,c1  a1 = tile(j=0) c2,c3  a2 = tile(j=1) c0,c1  a3 = tile(j=1) c2,c3 ----
    uint4 tr_h[2], tr_l[2], ti_h[2], ti_l[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      wfm_split(T[0][u][0][0], T[0][u][0][1], tr_h[u].x, tr_l[u].x);
      wfm_split(T[0][u][0][2], T[0][u][0][3], tr_h[u].y, tr_l[u].y);
      wfm_split(T[0][u][1][0], T[0][u][1][1], tr_h[u].z, tr_l[u].z);
      wfm_split(T[0][u][1][2], T[0][u][1][3], tr_h[u].w, tr_l[u].w);
      wfm_split(T[1][u][0][0], T[1][u][0][1], ti_h[u].x, ti_l[u].x);
      wfm_split(T[1][u][0][2], T[1][u][0][3], ti_h[u].y, ti_l[u].y);
      wfm_split(T[1][u][1][0], T[1][u][1][1], ti_h[u].z, ti_l[u].z);
      wfm_split(T[1][u][1][2], T[1][u][1][3], ti_h[u].w, ti_l[u].w);
    }

    // ---- stage 2 + |.|^2 + 2 x 2 binning: pix[u][b] is detector pixel (px(u), py(b)) of this lane ----
    float pix[2][4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint4 ch = s_c2[b * 2 + 0][lane];     // {Wr b0, Wr b1, Wi b0, Wi b1} hi
      const uint4 cl = s_c2[b * 2 + 1][lane];     // lo
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        float yr[4] = {0.f, 0.f, 0.f, 0.f}, yi[4] = {0.f, 0.f, 0.f, 0.f};
        uint4 nti_h, nti_l;
        nti_h.x = ti_h[u].x ^ 0x80008000u; nti_h.y = ti_h[u].y ^ 0x80008000u;
        nti_h.z = ti_h[u].z ^ 0x80008000u; nti_h.w = ti_h[u].w ^ 0x80008000u;
        nti_l.x = ti_l[u].x ^ 0x80008000u; nti_l.y = ti_l[u].y ^ 0x80008000u;
        nti_l.z = ti_l[u].z ^ 0x80008000u; nti_l.w = ti_l[u].w ^ 0x80008000u;
        // Yr = Tr.Wr - Ti.Wi
        wfm_mma(yr, tr_h[u], ch.x, ch.y);
        wfm_mma(yr, tr_l[u], ch.x, ch.y);
        wfm_mma(yr, nti_h, ch.z, ch.w);
        wfm_mma(yr, nti_l, ch.z, ch.w);
        // Yi = Tr.Wi + Ti.Wr
        wfm_mma(yi, tr_h[u], ch.z, ch.w);
        wfm_mma(yi, tr_l[u], ch.z, ch.w);
        wfm_mma(yi, ti_h[u], ch.x, ch.y);
        wfm_mma(yi, ti_l[u], ch.x, ch.y);
        if (PASS2_FULL) {
          wfm_mma(yr, tr_h[u], cl.x, cl.y);
          wfm_mma(yr, nti_h, cl.z, cl.w);
          wfm_mma(yi, tr_h[u], cl.z, cl.w);
          wfm_mma(yi, ti_h[u], cl.x, cl.y);
        }
        float i0 = fmaf(yr[0], yr[0], yi[0] * yi[0]) + fmaf(yr[1], yr[1], yi[1] * yi[1]);   // row g,   fy pair
        float i1 = fmaf(yr[2], yr[2], yi[2] * yi[2]) + fmaf(yr[3], yr[3], yi[3] * yi[3]);   // row g+8, fy pair
        i0 += __shfl_xor_sync(0xffffffffu, i0, 4);                                           // fx pair (g, g^1)
        i1 += __shfl_xor_sync(0xffffffffu, i1, 4);
        pix[u][b] = (g & 1) ? i1 : i0;
      }
    }

    // ---- flux normalisation, noise, centre of gravity ----
    float tot = 0.f;
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int b = 0; b < 4; ++b) tot += pix[u][b];
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, sft);
    const float scale = p.nphotons * p.flux[k] / tot;
    const uint32_t k0 = p.k0[e], k1 = p.k1[e];
    float s0 = 0.f, sx = 0.f, sy = 0.f;
    float* cube = p.bincube ? p.bincube + ((size_t)e * p.nvalid + k) * 256 : nullptr;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int px = 8 * (1 - u) + (g >> 1) + 4 * (g & 1);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int py = ((b < 2) ? 8 + 4 * b : 4 * (b - 2)) + q;
        const int pidx = py * 16 + px;
        float v = pix[u][b] * scale;
        v = aom_pixel_noise(v, p.noise, (uint32_t)(k * 256 + pidx), p.frame, p.wfs_index, k0, k1);
        if (cube) cube[pidx] = v;
        s0 += v;
        sx = fmaf(v, (float)px, sx);
        sy = fmaf(v, (float)py, sy);
      }
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
      sx += __shfl_xor_sync(0xffffffffu, sx, sft);
      sy += __shfl_xor_sync(0xffffffffu, sy, sft);
    }
    if (lane == 0) {
      const float gx = (s0 > 0.f) ? sx / s0 : p.cog_offset;
      const float gy = (s0 > 0.f) ? sy / s0 : p.cog_offset;
      float* sl = p.slopes + (size_t)e * p.lds;
      sl[k] = (gx - p.cog_offset) * p.pixsize;
      sl[p.nvalid + k] = (gy - p.cog_offset) * p.pixsize;
    }
    __syncwarp();
  }
}
