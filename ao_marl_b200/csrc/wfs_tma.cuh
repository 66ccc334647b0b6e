// Shack-Hartmann frame, third generation: TMA-staged screen tiles + register-resident tensor-pipe DFT.
//
// Same fused pipeline and the same arithmetic as wfs_frame_mma_kernel (wfs_mma.cuh) -- raytrace through the
// layers -> mirrors -> complex field -> pruned 2-D DFT as two chained fp16-split MMA stages -> |.|^2 ->
// 2 x 2 binning -> flux / noise -> centre of gravity, one warp per subaperture -- restructured around what
// ncu showed on B200 (profiles/r01_wfs_mma_E1024_*): 1780 warp instructions per subaperture, 30 % of them
// integer addressing, issue slots 43 % busy behind long-scoreboard stalls on the screen loads.
//
//   * every warp double-buffers the three 17 x 17 screen tiles of its NEXT subaperture in shared memory with one
//     3-D TMA box per layer (cp.async.bulk.tensor, box 24 x 17 x 1 of the [E][N][N] torus, starting at the
//     16-byte aligned column below the tile origin) completing on a
//     per-warp mbarrier, so the HBM latency overlaps the current subaperture's arithmetic; tiles that straddle
//     the torus seam (about 5 %) are filled by plain loads instead;
//   * lane (g, q) = (lane / 4, lane % 4) owns pixels rows {2g, 2g+1} x columns {4q .. 4q+3}: with the k / n
//     orderings of both MMA stages permuted accordingly (the permutations live in the constant twiddle
//     fragments) the field goes from the sincos straight into the B fragments of stage 1 -- no shared-memory
//     transpose -- and the 2 x 2 binning of stage 2 is entirely in-thread -- no shuffles;
//   * tile reads are 128-bit shared loads at immediate offsets of one base register;
//   * the mirror surface uses the 16-pixel pitch of the lattice: the separable stamp factors are two
//     [4][16] tables per CTA and the 4 x 4 actuator neighbourhood (plus the two tip-tilt volts) of the next
//     subaperture is prefetched one iteration ahead;
//   * the pupil mask is one byte per lane per subaperture.
//
// Eligibility is decided on the host (wfs_lattice_host.h); other geometries keep wfs_frame_mma_kernel.
// Replaces sutra's raytrace + fillcamplipup + cuFFT + abs2 + fillbincube + noise + centroid kernels behind
// WfsCompass.raytrace / compute_wfs_image / RtcCompass.do_centroids (shesha/supervisor/components/
// wfsCompass.py:334-343, sourceCompass.py:54-85, rtcCompass.py:557-563).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include "device_common.cuh"
#include "wfs_mma.cuh"
#include "wfs_lattice_host.h"

#define WFT_WARPS 8
#define WFT_MIN_CTAS 2
#define WFT_TILE_W 24                      // box width (floats): 17 needed, padded so that rows are 96 B apart
#define WFT_TILE_H 17
#define WFT_TILE_BYTES (WFT_TILE_W * WFT_TILE_H * 4)          // 1632 = bytes one box delivers
#define WFT_TILE_STRIDE 1664                                  // 13 x 128: TMA destinations stay 128-byte aligned
#define WFT_NG WFL_NG
#define WFT_MAX_LAYERS WFL_MAX_LAYERS

struct WfsFast {
  const uint2* sub;          // [nvalid] {y0 << 16 | x0, padded-lattice index of the neighbourhood origin}
  const short* amap;         // [GW * GW] actuator index or -1 (padded by WFL_PAD cells on every side)
  const unsigned char* pmask;// [nvalid][32] bit r*4+c = pupil(2g + r, 4q + c) of lane (g, q)
  const uint4* c1;           // [8][32]  stage-1 A fragments  [(mt*2 + part)*2 + hl][lane]
  const uint4* c2;           // [12][32] stage-2 B fragments  [b*3 + {hi, lo, -Wi}][lane]
  const float* fxy;          // [2][WFT_NG][16] separable stamp factor seen from a tile: x table then y table
  int GW;                    // side of the padded actuator map
  int sub_in_smem;           // stage the subaperture table in shared memory
  int* err;                  // device error word (bounded waits)
  long long items_per_cta;
};

struct WfsTmaParams {
  WfsParams p;
  WfsFast f;
  CUtensorMap maps[WFT_MAX_LAYERS];
};

__device__ __forceinline__ void wft_tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// Bilinear sample of one staged tile at this lane's 2 x 4 pixels.  The TMA box starts at the 16-byte aligned
// column below the tile origin (the inner coordinate of a tiled copy must be 16-byte aligned), so the wanted
// columns begin D = origin & 3 floats into the row; D is warp-uniform and resolved by a switch around this.
template <int D>
__device__ __forceinline__ void wft_layer(const float* __restrict__ t, const WfsLayer& L, float (&ph)[2][4]) {
  // four-tap form of the bilinear sample (weights per layer from the host): 4 FFMA per pixel and layer instead of
  // the 5 of the separable two-pass form; same value up to float rounding
  float v[3][8];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float4 a = *reinterpret_cast<const float4*>(t + r * WFT_TILE_W);
    v[r][0] = a.x; v[r][1] = a.y; v[r][2] = a.z; v[r][3] = a.w;
    if (D == 0) {
      v[r][4] = t[r * WFT_TILE_W + 4];
    } else {
      const float4 b = *reinterpret_cast<const float4*>(t + r * WFT_TILE_W + 4);
      v[r][4] = b.x; v[r][5] = b.y; v[r][6] = b.z; v[r][7] = b.w;
    }
  }
  const float w00 = L.w00, w01 = L.w01, w10 = L.w10, w11 = L.w11;
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float acc = ph[r][c];
      acc = fmaf(w00, v[r][D + c], acc);
      acc = fmaf(w01, v[r][D + c + 1], acc);
      acc = fmaf(w10, v[r + 1][D + c], acc);
      acc = fmaf(w11, v[r + 1][D + c + 1], acc);
      ph[r][c] = acc;
    }
}

// WFT_WARPS warps per CTA, two tile stages and two volt buffers per warp
template <int NL>
constexpr size_t wft_smem_bytes(int gw, int nvalid_smem) {
  return (size_t)WFT_WARPS * 2 * (NL > 0 ? NL : 1) * WFT_TILE_STRIDE + WFT_WARPS * 2 * 8 +
         8 * 32 * 16 + 12 * 32 * 16 + 256 * 4 + 2 * WFT_NG * 16 * 4 + WFT_WARPS * 2 * 32 * 4 +
         (((size_t)gw * gw * 2 + 15) & ~(size_t)15) + (size_t)nvalid_smem * 8;
}

// FULL = 1: three MMAs per product in both stages (fp32-grade); 0 drops the twiddle-lo pass of stage 2.
// The register allocation is bounded for WFT_WARPS warps per CTA and WFT_MIN_CTAS CTAs per SM.
template <int FULL, int NL>
__global__ void __launch_bounds__(WFT_WARPS * 32, WFT_MIN_CTAS) wfs_frame_tma_kernel(const __grid_constant__ WfsTmaParams P) {
  constexpr int NW = WFT_WARPS;
  const WfsParams& p = P.p;
  const WfsFast& f = P.f;
  extern __shared__ __align__(128) unsigned char wft_smem_raw[];
  unsigned char* sm = wft_smem_raw;
  constexpr int NLS = NL > 0 ? NL : 1;
  unsigned char* s_tiles = sm;                                             // [warp][stage][layer][WFT_TILE_STRIDE]
  uint64_t* s_bar = (uint64_t*)(s_tiles + (size_t)NW * 2 * NLS * WFT_TILE_STRIDE);   // [warp][stage]
  uint4* s_c1 = (uint4*)(s_bar + NW * 2);                                  // [8][32]
  uint4* s_c2 = s_c1 + 8 * 32;                                             // [12][32]
  float* s_half = (float*)(s_c2 + 12 * 32);                                // [256]
  float* s_fx = s_half + 256;                                              // [NG][16]
  float* s_fy = s_fx + WFT_NG * 16;                                        // [NG][16]
  float* s_vall = s_fy + WFT_NG * 16;                                      // [warp][stage][32]
  short* s_amap = (short*)(s_vall + NW * 2 * 32);
  uint2* s_sub = (uint2*)((unsigned char*)s_amap + ((f.GW * f.GW * 2 + 15) & ~15));

  // warp index through a shuffle: marks it (and the work-item index, tile coordinates, TMA operands derived from it)
  // warp-uniform for the compiler
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int g = lane >> 2, q = lane & 3;

  for (int i = threadIdx.x; i < 8 * 32; i += blockDim.x) s_c1[i] = f.c1[i];
  for (int i = threadIdx.x; i < 12 * 32; i += blockDim.x) s_c2[i] = f.c2[i];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_half[i] = p.halfxy[i];
  for (int i = threadIdx.x; i < 2 * WFT_NG * 16; i += blockDim.x) s_fx[i] = f.fxy[i];
  for (int i = threadIdx.x; i < f.GW * f.GW; i += blockDim.x) s_amap[i] = f.amap[i];
  if (f.sub_in_smem)
    for (int i = threadIdx.x; i < p.nvalid; i += blockDim.x) s_sub[i] = f.sub[i];
  if (threadIdx.x < NW * 2)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wft_smem_u32(s_bar + threadIdx.x)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const uint2* sub = f.sub_in_smem ? s_sub : f.sub;
  unsigned char* my_tiles = s_tiles + (size_t)warp * 2 * NLS * WFT_TILE_STRIDE;
  const uint32_t my_tiles_u32 = wft_smem_u32(my_tiles);
  const uint32_t my_bar_u32 = wft_smem_u32(s_bar + warp * 2);
  float* s_v = s_vall + warp * 2 * 32;
  const int lane_off = (2 * g) * WFT_TILE_W + 4 * q;         // floats, inside a tile

  const long long total = (long long)p.E * p.nvalid;
  const long long base = (long long)blockIdx.x * f.items_per_cta;
  long long end = base + f.items_per_cta;
  if (end > total) end = total;
  long long w = base + warp;
  if (w >= end) return;

  int e = (int)(w / p.nvalid), k = (int)(w % p.nvalid);
  int ring_e = -1;
  int rx[NLS], ry[NLS];                       // x0-independent part of the tile origin: (ix + ox[e]) mod N, (iy + oy[e]) mod N
  uint32_t phase_bits = 0;
  const int amap_lane = (lane >> 2) * f.GW + (lane & 3);
  const int tt_lane = (2 * g + p.tt_off) * p.tt_dim + 4 * q + p.tt_off;      // this lane's pixel (2g, 4q) in the tip-tilt planes
  const float* const tt_plane1 = p.tt_planes + (size_t)p.tt_dim * p.tt_dim;

  // ---- prefetch of one work item into `stage`: TMA boxes, neighbourhood volts, pupil byte ----
  uint32_t n_xy = 0, n_pm = 0, n_d = 0;      // n_d: 2 bits per layer = tile origin column & 3
  float n_v = 0.f;
  bool n_seam = false;
  auto prefetch = [&](int pe, int pk, int stage) {
    uint2 sb = sub[pk];
    sb.x = __shfl_sync(0xffffffffu, sb.x, 0); sb.y = __shfl_sync(0xffffffffu, sb.y, 0);
    n_xy = sb.x;
    if (NL > 0) {
      if (pe != ring_e) {
#pragma unroll
        for (int l = 0; l < NL; ++l) {
          const int N = p.layer[l].N;
          int a = p.layer[l].ix + p.layer[l].ox[pe];  a -= (a >= N) ? N : 0;
          int b = p.layer[l].iy + p.layer[l].oy[pe];  b -= (b >= N) ? N : 0;
          rx[l] = a; ry[l] = b;
        }
        ring_e = pe;
      }
      const int x0 = (int)(sb.x & 0xffffu), y0 = (int)(sb.x >> 16);
      int tc[NLS], tr[NLS];
      bool seam = false;
      uint32_t dbits = 0;
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        const int N = p.layer[l].N;
        int c = x0 + rx[l];  c -= (c >= N) ? N : 0;
        int r = y0 + ry[l];  r -= (r >= N) ? N : 0;
        tc[l] = c & ~3; tr[l] = r;
        dbits |= (uint32_t)(c & 3) << (2 * l);
        seam |= (c + WFT_TILE_H > N) | (r + WFT_TILE_H > N);
      }
      n_seam = seam;
      n_d = dbits;
      if (!seam) {
        // the stage was read (or, on the seam path, written) through the generic proxy: order those accesses before the
        // async-proxy writes of the new boxes
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
      }
      if (!seam && lane == 0) {
        const uint32_t bar = my_bar_u32 + stage * 8;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(NL * WFT_TILE_BYTES) : "memory");
#pragma unroll
        for (int l = 0; l < NL; ++l)
          wft_tma_load_3d(my_tiles_u32 + (stage * NL + l) * WFT_TILE_STRIDE, &P.maps[l], tc[l], tr[l], pe, bar);
      }
    }
    n_v = 0.f;
    if (p.use_dm && lane < 18) {
      int idx = (lane < 16) ? (int)s_amap[(int)sb.y + amap_lane] : p.pzt_nact + lane - 16;
      if (idx >= 0) n_v = __ldg(p.volts + (size_t)pe * p.ldv + idx);
    }
    n_pm = f.pmask[(size_t)pk * 32 + lane];
  };

  prefetch(e, k, 0);
  s_v[lane] = n_v;
  __syncwarp();
  for (int it = 0; w < end; ++it, w += NW) {
    const int s = it & 1;                       // stage of the current item
    const uint32_t c_xy = n_xy, c_pm = n_pm, c_d = n_d;
    const bool c_seam = n_seam;
    const int ce = e, ck = k;
    const int x0 = (int)(c_xy & 0xffffu), y0 = (int)(c_xy >> 16);

    // ---- next work item ----
    const bool has_next = (w + NW) < end;
    if (has_next) {
      k += NW;
      if (k >= p.nvalid) { k -= p.nvalid; e += 1; }
      prefetch(e, k, s ^ 1);
    }

    // ---- static planes of the current subaperture (L2-resident tables), issued before the wait ----
    float4 tta[2], ttb[2];
    if (p.use_dm) {
      const int to = y0 * p.tt_dim + x0 + tt_lane;
      tta[0] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to));
      tta[1] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to + p.tt_dim));
      ttb[0] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to));
      ttb[1] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to + p.tt_dim));
    }

    float ph[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) ph[r][c] = 0.f;

    // ---- atmosphere: bilinear sample of the staged tiles ----
    if (NL > 0) {
      if (!c_seam) {
        wft_mbar_wait(my_bar_u32 + s * 8, (phase_bits >> s) & 1u, f.err);
        phase_bits ^= (1u << s);
      } else {
        // tile straddles the torus seam: fill the stage with wrapped plain loads
#pragma unroll 1
        for (int l = 0; l < NL; ++l) {
          const int N = p.layer[l].N;
          const float* scr = p.layer[l].screen + (size_t)ce * N * N;
          int c0 = x0 + p.layer[l].ix + p.layer[l].ox[ce];  c0 -= (c0 >= N) ? N : 0;  c0 -= (c0 >= N) ? N : 0;
          int r0 = y0 + p.layer[l].iy + p.layer[l].oy[ce];  r0 -= (r0 >= N) ? N : 0;  r0 -= (r0 >= N) ? N : 0;
          float* tile = reinterpret_cast<float*>(my_tiles + (s * NL + l) * WFT_TILE_STRIDE);
          for (int i = lane; i < WFT_TILE_H * WFT_TILE_H; i += 32) {
            const int r = i / WFT_TILE_H, c = i - r * WFT_TILE_H;
            int rr = r0 + r;  rr -= (rr >= N) ? N : 0;
            int cc = c0 + c;  cc -= (cc >= N) ? N : 0;
            tile[r * WFT_TILE_W + (c0 & 3) + c] = __ldg(scr + (size_t)rr * N + cc);
          }
        }
        __syncwarp();
      }
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        const float* t = reinterpret_cast<const float*>(my_tiles + (s * NL + l) * WFT_TILE_STRIDE) + lane_off;
        switch ((c_d >> (2 * l)) & 3u) {
          case 0: wft_layer<0>(t, p.layer[l], ph); break;
          case 1: wft_layer<1>(t, p.layer[l], ph); break;
          case 2: wft_layer<2>(t, p.layer[l], ph); break;
          default: wft_layer<3>(t, p.layer[l], ph); break;
        }
      }
    }

    // ---- mirrors: separable stamps of the 4 x 4 lattice neighbourhood + two tip-tilt planes ----
    if (p.use_dm) {
      const float* V = s_v + s * 32;
      float u[2][WFT_NG];
#pragma unroll
      for (int jx = 0; jx < WFT_NG; ++jx) u[0][jx] = u[1][jx] = 0.f;
#pragma unroll
      for (int jy = 0; jy < WFT_NG; ++jy) {
        const float4 vr = *reinterpret_cast<const float4*>(V + jy * 4);
        const float2 fyv = *reinterpret_cast<const float2*>(s_fy + jy * 16 + 2 * g);
        u[0][0] = fmaf(fyv.x, vr.x, u[0][0]); u[0][1] = fmaf(fyv.x, vr.y, u[0][1]);
        u[0][2] = fmaf(fyv.x, vr.z, u[0][2]); u[0][3] = fmaf(fyv.x, vr.w, u[0][3]);
        u[1][0] = fmaf(fyv.y, vr.x, u[1][0]); u[1][1] = fmaf(fyv.y, vr.y, u[1][1]);
        u[1][2] = fmaf(fyv.y, vr.z, u[1][2]); u[1][3] = fmaf(fyv.y, vr.w, u[1][3]);
      }
      float dm[2][4];
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) dm[r][c] = 0.f;
#pragma unroll
      for (int jx = 0; jx < WFT_NG; ++jx) {
        const float4 fxv = *reinterpret_cast<const float4*>(s_fx + jx * 16 + 4 * q);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          dm[r][0] = fmaf(u[r][jx], fxv.x, dm[r][0]);
          dm[r][1] = fmaf(u[r][jx], fxv.y, dm[r][1]);
          dm[r][2] = fmaf(u[r][jx], fxv.z, dm[r][2]);
          dm[r][3] = fmaf(u[r][jx], fxv.w, dm[r][3]);
        }
      }
      const float tt0 = V[16], tt1 = V[17];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        ph[r][0] += fmaf(tt1, ttb[r].x, fmaf(tt0, tta[r].x, dm[r][0]));
        ph[r][1] += fmaf(tt1, ttb[r].y, fmaf(tt0, tta[r].y, dm[r][1]));
        ph[r][2] += fmaf(tt1, ttb[r].z, fmaf(tt0, tta[r].z, dm[r][2]));
        ph[r][3] += fmaf(tt1, ttb[r].w, fmaf(tt0, tta[r].w, dm[r][3]));
      }
    }

    // ---- complex field -> fp16 hi / lo B fragments of stage 1 (row 2g + j feeds n-tile j) ----
    uint32_t xr_h[2][2], xr_l[2][2], xi_h[2][2], xi_l[2][2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const float4 hf = *reinterpret_cast<const float4*>(s_half + (2 * g + r) * 16 + 4 * q);
      const float hv[4] = {hf.x, hf.y, hf.z, hf.w};
      float re[4], im[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float sn, cs;
        wfm_sincos(p.k2 * ph[r][c] - hv[c], sn, cs);
        const bool on = (c_pm >> (r * 4 + c)) & 1u;
        re[c] = on ? cs : 0.f;
        im[c] = on ? sn : 0.f;
      }
      wfm_split(re[0], re[1], xr_h[r][0], xr_l[r][0]);
      wfm_split(re[2], re[3], xr_h[r][1], xr_l[r][1]);
      wfm_split(im[0], im[1], xi_h[r][0], xi_l[r][0]);
      wfm_split(im[2], im[3], xi_h[r][1], xi_l[r][1]);
    }

    // ---- stage 1: T[part][mt][j] (16 x 8 tiles: rows = kept fx (pair-interleaved), cols = y) ----
    // Issue order = source order (asm volatile): the eight accumulator tiles advance in lock step, so eight
    // independent MMAs are in flight and the ~30-cycle MMA latency of a dependent chain is covered.
    float T[2][2][2][4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int c = 0; c < 4; ++c) T[a][mt][j][c] = 0.f;
    {
      uint32_t nxi_h[2][2], nxi_l[2][2];
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int c = 0; c < 2; ++c) { nxi_h[j][c] = xi_h[j][c] ^ 0x80008000u; nxi_l[j][c] = xi_l[j][c] ^ 0x80008000u; }
      uint4 wr_h[2], wr_l[2], wi_h[2], wi_l[2];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        wr_h[mt] = s_c1[(mt * 4 + 0) * 32 + lane]; wr_l[mt] = s_c1[(mt * 4 + 1) * 32 + lane];
        wi_h[mt] = s_c1[(mt * 4 + 2) * 32 + lane]; wi_l[mt] = s_c1[(mt * 4 + 3) * 32 + lane];
      }
#define WFT_S1(WR, WI, XR, XI, NXI)                                            \
  _Pragma("unroll") for (int mt = 0; mt < 2; ++mt)                             \
  _Pragma("unroll") for (int j = 0; j < 2; ++j) {                              \
    wfm_mma(T[0][mt][j], WR[mt], XR[j][0], XR[j][1]);                          \
    wfm_mma(T[1][mt][j], WI[mt], XR[j][0], XR[j][1]);                          \
  }                                                                            \
  _Pragma("unroll") for (int mt = 0; mt < 2; ++mt)                             \
  _Pragma("unroll") for (int j = 0; j < 2; ++j) {                              \
    wfm_mma(T[0][mt][j], WI[mt], NXI[j][0], NXI[j][1]);                        \
    wfm_mma(T[1][mt][j], WR[mt], XI[j][0], XI[j][1]);                          \
  }
      // Tr = Wr.Xr - Wi.Xi     Ti = Wi.Xr + Wr.Xi     (hi.hi, hi.lo, lo.hi)
      WFT_S1(wr_h, wi_h, xr_h, xi_h, nxi_h)
      WFT_S1(wr_h, wi_h, xr_l, xi_l, nxi_l)
      WFT_S1(wr_l, wi_l, xr_h, xi_h, nxi_h)
#undef WFT_S1
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

    // ---- stage 2 + |.|^2 + 2 x 2 binning, all in-thread: pix[u][b] = detector pixel (px(u, g), py(b, q)) ----
    // Four accumulator tiles (Yr / Yi of both fx tiles) advance in lock step per fy tile b.
    float pix[2][4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint4 ch = s_c2[(b * 3 + 0) * 32 + lane];     // {Wr b0, Wr b1, Wi b0, Wi b1} hi
      const uint4 cn = s_c2[(b * 3 + 2) * 32 + lane];     // {-Wi_hi b0, -Wi_hi b1, -Wi_lo b0, -Wi_lo b1}
      uint4 cl = make_uint4(0u, 0u, 0u, 0u);
      if (FULL) cl = s_c2[(b * 3 + 1) * 32 + lane];       // lo
      float yr[2][4], yi[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int c = 0; c < 4; ++c) { yr[u][c] = 0.f; yi[u][c] = 0.f; }
      {
        // Yr = Tr.Wr - Ti.Wi     Yi = Tr.Wi + Ti.Wr
#pragma unroll
        for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], tr_h[u], ch.x, ch.y); wfm_mma(yi[u], tr_h[u], ch.z, ch.w); }
#pragma unroll
        for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], ti_h[u], cn.x, cn.y); wfm_mma(yi[u], ti_h[u], ch.x, ch.y); }
#pragma unroll
        for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], tr_l[u], ch.x, ch.y); wfm_mma(yi[u], tr_l[u], ch.z, ch.w); }
#pragma unroll
        for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], ti_l[u], cn.x, cn.y); wfm_mma(yi[u], ti_l[u], ch.x, ch.y); }
        if (FULL) {
#pragma unroll
          for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], tr_h[u], cl.x, cl.y); wfm_mma(yi[u], tr_h[u], cl.z, cl.w); }
#pragma unroll
          for (int u = 0; u < 2; ++u) { wfm_mma(yr[u], ti_h[u], cn.z, cn.w); wfm_mma(yi[u], ti_h[u], cl.x, cl.y); }
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        float a = yr[u][0] * yr[u][0];
        a = fmaf(yi[u][0], yi[u][0], a);
        a = fmaf(yr[u][1], yr[u][1], a);
        a = fmaf(yi[u][1], yi[u][1], a);
        float c = yr[u][2] * yr[u][2];
        c = fmaf(yi[u][2], yi[u][2], c);
        c = fmaf(yr[u][3], yr[u][3], c);
        c = fmaf(yi[u][3], yi[u][3], c);
        pix[u][b] = a + c;
      }
    }

    // ---- flux normalisation, noise, centre of gravity ----
    const bool plain = (p.noise < 0.f) && (p.bincube == nullptr);     // centre of gravity is scale invariant
    float s0 = 0.f, sx = 0.f, sy = 0.f;
    if (plain) {
      const float r0 = (pix[0][0] + pix[0][1]) + (pix[0][2] + pix[0][3]);   // px = 8 + g
      const float r1 = (pix[1][0] + pix[1][1]) + (pix[1][2] + pix[1][3]);   // px = g
      s0 = r0 + r1;
      sx = fmaf(r0, (float)(8 + g), r1 * (float)g);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int py = ((b < 2) ? 8 + 4 * b : 4 * (b - 2)) + q;
        sy = fmaf(pix[0][b] + pix[1][b], (float)py, sy);
      }
    } else {
      float tot = 0.f;
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int b = 0; b < 4; ++b) tot += pix[u][b];
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, sft);
      const float scale = p.nphotons * p.flux[ck] / tot;
      const uint32_t k0 = p.k0[ce], k1 = p.k1[ce];
      float* cube = p.bincube ? p.bincube + ((size_t)ce * p.nvalid + ck) * 256 : nullptr;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int px = 8 * (1 - u) + g;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int py = ((b < 2) ? 8 + 4 * b : 4 * (b - 2)) + q;
          const int pidx = py * 16 + px;
          float v = pix[u][b] * scale;
          v = aom_pixel_noise(v, p.noise, (uint32_t)(ck * 256 + pidx), p.frame, p.wfs_index, k0, k1);
          if (cube) cube[pidx] = v;
          s0 += v;
          sx = fmaf(v, (float)px, sx);
          sy = fmaf(v, (float)py, sy);
        }
      }
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
      sx += __shfl_xor_sync(0xffffffffu, sx, sft);
      sy += __shfl_xor_sync(0xffffffffu, sy, sft);
    }
    if (lane == 0) {
      const float inv = __frcp_rn(s0);
      const float gx = (s0 > 0.f) ? sx * inv : p.cog_offset;
      const float gy = (s0 > 0.f) ? sy * inv : p.cog_offset;
      float* sl = p.slopes + (size_t)ce * p.lds;
      sl[ck] = (gx - p.cog_offset) * p.pixsize;
      sl[p.nvalid + ck] = (gy - p.cog_offset) * p.pixsize;
    }
    // ---- hand the prefetched neighbourhood volts to the next iteration ----
    if (has_next) s_v[(s ^ 1) * 32 + lane] = n_v;
    __syncwarp();
  }
}
