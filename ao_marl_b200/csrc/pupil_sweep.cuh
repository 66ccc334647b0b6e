// pupil_sweep.cuh -- one pass over the pupil-plane phase of every environment without materialising it.
//
// Two consumers share the sweep:
//   MODE 0  geometric controller (RlSupervisor.next_part_one_geo, shesha/supervisor/rlSupervisor.py:989-1013; sutra
//           comp_dphi + the sparse IF product of comp_com): target phase through the atmosphere, masked by the pupil,
//           projected on the lattice columns (T[e][y][gx], see geo_kernels.cuh) + the pupil sums of the piston /
//           tip-tilt rows;
//   MODE 1  target Strehl (TargetCompass.comp_tar_image / comp_strehl, shesha/supervisor/components/targetCompass.py:139-196,
//           atmosphere + mirrors, pupil sums of m, m phi, m phi^2 (variance) and of m exp(i k phi): the on-axis
//           intensity |<exp(i k phi)>|^2 is the peak of the PSF the reference's FFT would give for a tilt-free residual.
//   MODE 2  MODE 1 + the 3 x 3 central pixels of that PSF on the reference's focal grid (zero-padded FFT of size Nfft:
//           pixel (a, b) = |sum m exp(i k phi) exp(-2 pi i (a x + b y) / Nfft)|^2), by direct summation: the brightest
//           pixel and its neighbours are what the reference's comp_strehl(do_fit=True) looks at in closed loop.
//           Separable twiddles: per pixel four products with the lane's constant column twiddles, per row twelve with
//           the row twiddle (16 more accumulators, no second pass).
//
// Layout of the work.  A warp owns a 128-pixel column block of a strip of consecutive pupil rows of one environment:
// one lane = four pixels of the current row.  Pupil row y needs the screen rows r(y), r(y)+1 of every layer, and
// r(y)+1 = r(y+1): the warp keeps a three-slot ring of staged screen-row segments (136 floats per layer) in shared
// memory, filled two rows ahead by 1-D bulk copies (cp.async.bulk, completion on a per-slot mbarrier), so each screen
// row is fetched once per strip with no address arithmetic in the lanes, and 6 KB of shared memory per warp leave 32
// warps per SM.  (A first version staged whole 656-float rows per warp: 28 KB per warp, 8 warps per SM, issue slots
// 20 % busy -- profiles/r01_pupil_sweep_v1_*.)  Copies start at the 16-byte aligned column below the wanted one (bulk
// copies need 16-byte alignment; a segment wraps around the torus in at most two pieces); the residual offset
// D = column & 3 is warp-uniform and resolved by a switch, so the lanes read the staged rows with aligned LDS.128:
// 4 vector loads + 16 FFMA per layer for four pixels (four-tap bilinear weights from the host).
// Pixels are addressed in the lattice frame x' = x - (i1_0 - pzt_off) (>= 0): a column block is eight 16-pixel lattice
// chunks, and the pupil mask / tip-tilt planes are repacked once into that frame (sweep_tables_kernel).
// MODE 0 row pass: Q[j][u] = sum_k f[16u+k] row[16j+k] is one FFMA chain per lane (32 = 8 chunks x 4 offsets); the
// lattice sums T[g] = Q[g][0] + Q[g+1][1] + Q[g+2][2] + Q[g+3][3] reach three chunks to the right, so every block
// writes its 11 partial sums (g = 8 cb - 3 .. 8 cb + 7) to Tp[e][y][cb][12] and geo_cols_kernel adds the two
// blocks that can contribute to a lattice column -- no atomics, deterministic.
#pragma once
#include "device_common.cuh"
#include "pupil_kernels.cuh"

#define PSW_WARPS 8
#define PSW_SLOTS 3
#define PSW_STRIP 46        // pupil rows per warp: 644 = 14 x 46 on the 40x40 grid
#define PSW_BW 136          // staged floats per layer and screen row: 128 pixels + 1, rounded to 16 bytes, + alignment slack
#define PSW_TP 12           // partial lattice sums per block and row (11 used)
#define PSW_MOM2 24         // doubles per environment of the MODE 2 sums (21 used)

struct SweepParams {
  WfsParams w;
  const uint32_t* maskw;    // [n][32 nb]     pupil mask, one byte per pixel, four per word (lattice frame, 0 outside)
  const float* ttp;         // [2][n][128 nb] tip-tilt planes in the lattice frame, zero outside the pupil frame
  float* Tp;                // MODE 0: [E][n][nb][PSW_TP]
  double* mom;              // MODE 0: [E][4] sums of m phi, m phi tt_x, m phi tt_y
                            // MODE 1: [E][5] sums of m, m phi, m phi^2, m cos(k phi), m sin(k phi)
                            // MODE 2: [E][PSW_MOM2]: the five above, then T1..T4 of a = -1, 0, +1 and (Re, Im) of
                            //         (a, b) = (-1, 0), (+1, 0)  (see psw_core_pixels)
  float k2t;                // MODE 1: 2 pi / target wavelength
  float core_step;          // MODE 2: 1 / Nfft (turns of the focal twiddle per pupil pixel)
  int nb;                   // column blocks per row
  int n_strips;
  int* err;
};

__host__ __device__ inline size_t psw_warp_floats(int NL) {
  return (size_t)PSW_SLOTS * NL * PSW_BW + 160 + 32 + 48 + 16 + 8;   // ring, out row, Q, volt window, R row, barriers
}
__host__ __device__ inline size_t psw_smem_bytes(int NL, bool pe = false) {
  return (PSW_WARPS * psw_warp_floats(NL) + 64) * sizeof(float) + (pe ? (size_t)NL * sizeof(WindRec) : 0);
}

// mask / tip-tilt planes in the lattice frame; grid (n), block 128
__global__ void sweep_tables_kernel(WfsParams p, uint32_t* maskw, float* ttp, int nb) {
  const int y = blockIdx.x;
  const int xs0 = p.i1_0 - p.pzt_off;
  for (int m = threadIdx.x; m < 32 * nb; m += blockDim.x) {
    uint32_t word = 0;
    for (int c = 0; c < 4; ++c) {
      const int x = 4 * m + c + xs0;
      const bool in = x >= 0 && x < p.n;
      const bool lit = in && p.mpupil[(size_t)y * p.n + x] != 0.f;
      word |= (lit ? 1u : 0u) << (8 * c);
      for (int j = 0; j < 2; ++j) {
        float v = 0.f;
        if (in && p.tt_planes)
          v = p.tt_planes[(size_t)j * p.tt_dim * p.tt_dim + (size_t)(y + p.tt_off) * p.tt_dim + x + p.tt_off];
        ttp[((size_t)j * p.n + y) * 128 * nb + 4 * m + c] = v;
      }
    }
    maskw[(size_t)y * 32 * nb + m] = word;
  }
}

__device__ __forceinline__ void psw_bulk(uint32_t dst, const float* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// four pixels of one layer from the staged upper / lower screen rows (16-byte aligned pointers, wanted columns start
// D floats in)
template <int D, class Wt>      // Wt: WfsLayer (common offset) or WindRec (the environment's own)
__device__ __forceinline__ void psw_layer(const float* __restrict__ up, const float* __restrict__ lo, const Wt& L,
                                          float (&ph)[4]) {
  float a[8], b[8];
  const float4 a0 = *reinterpret_cast<const float4*>(up), b0 = *reinterpret_cast<const float4*>(lo);
  a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
  b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
  if (D == 0) {
    a[4] = up[4]; b[4] = lo[4];
  } else {
    const float4 a1 = *reinterpret_cast<const float4*>(up + 4), b1 = *reinterpret_cast<const float4*>(lo + 4);
    a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
    b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
  }
  const float w00 = L.w00, w01 = L.w01, w10 = L.w10, w11 = L.w11;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float acc = ph[c];
    acc = fmaf(w00, a[D + c], acc);
    acc = fmaf(w01, a[D + c + 1], acc);
    acc = fmaf(w10, b[D + c], acc);
    acc = fmaf(w11, b[D + c + 1], acc);
    ph[c] = acc;
  }
}

// PE: per-environment winds -- the block's environment reads its layer offsets from P.w.wind once, into shared memory
template <int NL, int MODE, bool PE = false>
__global__ void __launch_bounds__(PSW_WARPS * 32, MODE == 2 ? 3 : 4) pupil_sweep_kernel(const __grid_constant__ SweepParams P) {
  extern __shared__ __align__(128) float psw_smem[];
  const WfsParams& p = P.w;
  // the warp index through a shuffle: the compiler then keeps everything derived from it (strip, column block, the
  // source pointers of the bulk copies) in uniform registers instead of broadcasting it per copy
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int e = blockIdx.y;
  const int nl = p.n_layers < NL ? p.n_layers : NL;

  float* s_f = psw_smem;                                    // [64] stamp taps, zero beyond ss
  float* ring = psw_smem + 64 + (size_t)warp * psw_warp_floats(NL);   // [PSW_SLOTS][NL][PSW_BW]
  float* s_out = ring + PSW_SLOTS * NL * PSW_BW;            // [8][20]   MODE 0: masked phase of the row, lattice chunks
  float* s_q = s_out + 160;                                 // [8][4]    MODE 0: chunk partial sums
  float* s_v = s_q + 32;                                    // [4][12]   MODE 1: volts of the four lattice rows in reach
  float* s_r = s_v + 48;                                    // [16]      MODE 1: R_y[g], g = 8 cb - 3 + index
  unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_r + 16);   // [PSW_SLOTS]
  WindRec* s_wr = reinterpret_cast<WindRec*>(psw_smem + 64 + PSW_WARPS * psw_warp_floats(NL));   // PE: [NL] this environment's offsets

  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_f[i] = i < p.ss ? p.stamp1d[i] : 0.f;
  if (PE && threadIdx.x < 8 * nl)
    reinterpret_cast<uint32_t*>(s_wr)[threadIdx.x] =
        __ldg(reinterpret_cast<const uint32_t*>(p.wind + (size_t)(threadIdx.x >> 3) * p.E + e) + (threadIdx.x & 7));
  if (lane < 16) s_r[lane] = 0.f;
  if (lane < PSW_SLOTS)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wft_smem_u32(s_bar + lane)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const int item = blockIdx.x * PSW_WARPS + warp;
  if (item >= P.n_strips * P.nb) return;
  const int strip = item / P.nb, cb = item - strip * P.nb;
  const int yb = strip * PSW_STRIP;
  const int rows = min(PSW_STRIP, p.n - yb);
  const int xs0 = p.i1_0 - p.pzt_off, ys0 = p.j1_0 - p.pzt_off;

  // per layer: source of the next screen row to fetch (segment start, 16-byte aligned), rows left before the torus
  // wraps, length of the first piece, residual column offset
  const float* src[NL];
  int left[NL], len0[NL], dd[NL];
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    src[l] = nullptr; left[l] = len0[l] = dd[l] = 0;
    if (l < nl) {
      const WfsLayer& L = p.layer[l];
      const int N = L.N;
      const int oy = __shfl_sync(0xffffffffu, __ldg(L.oy + e), 0), ox = __shfl_sync(0xffffffffu, __ldg(L.ox + e), 0);
      const int ix = PE ? s_wr[l].ix : L.ix, iy = PE ? s_wr[l].iy : L.iy;
      int r = yb + iy + oy; r -= (r >= N) ? N : 0;
      int c = (128 * cb + xs0 + ix + ox) % N;             // column of the block's first pixel (x may lie outside the frame)
      c += (c < 0) ? N : 0;
      dd[l] = c & 3; c &= ~3;
      src[l] = L.screen + (size_t)e * N * N + c + (size_t)r * N;
      left[l] = N - r;
      len0[l] = min(PSW_BW, N - c) * 4;
    }
  }
  const uint32_t ring_u32 = wft_smem_u32(ring), bar_u32 = wft_smem_u32(s_bar);

  // every lane keeps the (warp-uniform) copy state, lane 0 alone issues: the state then lives in uniform registers
  auto issue = [&](int slot) {        // next screen row of every layer -> ring slot
    const uint32_t bar = bar_u32 + 8 * slot;
    if (lane == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(nl * PSW_BW * 4) : "memory");
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      if (l < nl) {
        const uint32_t dst = ring_u32 + (uint32_t)((slot * NL + l) * PSW_BW) * 4u;
        if (lane == 0) {
          psw_bulk(dst, src[l], (uint32_t)len0[l], bar);
          if (len0[l] < PSW_BW * 4)    // the segment wraps: the rest starts at column 0 of the same screen row
            psw_bulk(dst + (uint32_t)len0[l], src[l] - (p.layer[l].N - len0[l] / 4), (uint32_t)(PSW_BW * 4 - len0[l]), bar);
        }
        src[l] += p.layer[l].N;
        if (--left[l] == 0) { src[l] -= (size_t)p.layer[l].N * p.layer[l].N; left[l] = p.layer[l].N; }
      }
    }
  };

  if (nl > 0) {
    for (int i = 0; i < 3 && i <= rows; ++i) issue(i);
  }
  int s_up = 0, s_lo = 1;                           // ring slots of the upper / lower screen rows of the current pupil row
  uint32_t par_lo = 0;                              // phase parity the lower slot completes next

  // MODE 0: s1 = sum v, s2 = sum v ttx, s3 = sum v tty ; MODE 1: s0 = count, s1 = sum v, s2 = sum v^2, s3 / s4 = sum cos / sin (k v)
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, s4 = 0.f;
  float tt0 = 0.f, tt1 = 0.f;
  const float* volts = nullptr;
  const bool dm = MODE >= 1 && p.use_dm;
  if (dm) {
    volts = p.volts + (size_t)e * p.ldv;
    tt0 = __ldg(volts + p.pzt_nact); tt1 = __ldg(volts + p.pzt_nact + 1);
  }
  // MODE 2: column twiddles of this lane's four pixels (any origin: a shift of the pupil is a phase factor of the focal
  // amplitude) and the sums T1..T4 = sum_rows (Re cy, Im sy, Im cy, Re sy) of the three row amplitudes R_a
  float cxw[4], sxw[4], tc[3][4], tz[4];
  if (MODE == 2) {
#pragma unroll
    for (int c = 0; c < 4; ++c) sincospif(2.f * (float)(128 * cb + 4 * lane + c) * P.core_step, &sxw[c], &cxw[c]);
#pragma unroll
    for (int a = 0; a < 3; ++a) { tc[a][0] = tc[a][1] = tc[a][2] = tc[a][3] = 0.f; }
    tz[0] = tz[1] = tz[2] = tz[3] = 0.f;
  }
  // row twiddle exp(2 pi i y / Nfft), advanced by a rotation per row (46 rows per strip: the recurrence stays at 1e-6)
  float cyw = 1.f, syw = 0.f, cdw = 1.f, sdw = 0.f;
  if (MODE == 2) {
    sincospif(2.f * (float)yb * P.core_step, &syw, &cyw);
    sincospif(2.f * P.core_step, &sdw, &cdw);
  }
  float fq[16];                                    // MODE 0: the 16 taps of this lane's lattice offset u = lane & 3
  if (MODE == 0) {
#pragma unroll
    for (int k = 0; k < 16; ++k) fq[k] = s_f[16 * (lane & 3) + k];
  }
  const int ngw = 32 * P.nb, ga = 32 * cb + lane;   // groups per row of the tables, this lane's group
  const int jl = lane >> 2, k0 = 4 * (lane & 3);    // lattice chunk inside the block, first pixel inside the chunk
  int ro = yb * ngw + ga;                           // this lane's group in the mask / tip-tilt tables, current row
  const float4* ttp4 = reinterpret_cast<const float4*>(P.ttp);
  const int ty_off = p.n * ngw;
  float* tp = MODE == 0 ? P.Tp + (((size_t)e * p.n + yb) * P.nb + cb) * PSW_TP + lane : nullptr;
  int jy = (yb - ys0) >> 4, ky = (yb - ys0) & 15;
  bool new_jy = true;

  for (int i = 0; i < rows; ++i) {
    const uint32_t mask = __ldg(P.maskw + ro);
    float4 tx = make_float4(0.f, 0.f, 0.f, 0.f), ty = tx;
    if (mask != 0u && (MODE == 0 || dm)) { tx = __ldg(ttp4 + ro); ty = __ldg(ttp4 + ro + ty_off); }
    ro += ngw;
    if (dm) {
      // R_y[g] = sum_u f[16 u + ky] v[jy - u][g] over the at most four lattice rows whose stamp covers this pupil row
      if (new_jy) {
        new_jy = false;
        if (lane < 11) {
          const int g = 8 * cb - 3 + lane;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int gy = jy - u;
            float v = 0.f;
            if (g >= 0 && g < p.grid_n && gy >= 0 && gy < p.grid_n) {
              const int a = __ldg(p.act_map + gy * p.grid_n + g);
              if (a >= 0) v = __ldg(volts + a);
            }
            s_v[12 * u + lane] = v;
          }
        }
        __syncwarp();
      }
      if (lane < 11) {
        float r = 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u) r = fmaf(s_f[16 * u + ky], s_v[12 * u + lane], r);
        s_r[lane] = r;
      }
      __syncwarp();
      if (++ky == 16) { ky = 0; ++jy; new_jy = true; }
    }
    if (nl > 0) {
      if (i == 0 && !wft_mbar_wait(bar_u32, 0, P.err)) return;
      if (!wft_mbar_wait(bar_u32 + 8 * s_lo, par_lo, P.err)) return;
    }
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (mask != 0u) {
      const float* up = ring + (s_up * NL) * PSW_BW + 4 * lane;
      const float* lo = ring + (s_lo * NL) * PSW_BW + 4 * lane;
      float ph[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        if (l < nl) {
          if (PE) {
            switch (dd[l]) {
              case 0: psw_layer<0>(up + l * PSW_BW, lo + l * PSW_BW, s_wr[l], ph); break;
              case 1: psw_layer<1>(up + l * PSW_BW, lo + l * PSW_BW, s_wr[l], ph); break;
              case 2: psw_layer<2>(up + l * PSW_BW, lo + l * PSW_BW, s_wr[l], ph); break;
              default: psw_layer<3>(up + l * PSW_BW, lo + l * PSW_BW, s_wr[l], ph); break;
            }
          } else {
            switch (dd[l]) {
              case 0: psw_layer<0>(up + l * PSW_BW, lo + l * PSW_BW, p.layer[l], ph); break;
              case 1: psw_layer<1>(up + l * PSW_BW, lo + l * PSW_BW, p.layer[l], ph); break;
              case 2: psw_layer<2>(up + l * PSW_BW, lo + l * PSW_BW, p.layer[l], ph); break;
              default: psw_layer<3>(up + l * PSW_BW, lo + l * PSW_BW, p.layer[l], ph); break;
            }
          }
        }
      }
      if (dm) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float r = s_r[jl - u + 3];
          const float4 f4 = *reinterpret_cast<const float4*>(s_f + 16 * u + k0);
          ph[0] = fmaf(r, f4.x, ph[0]); ph[1] = fmaf(r, f4.y, ph[1]);
          ph[2] = fmaf(r, f4.z, ph[2]); ph[3] = fmaf(r, f4.w, ph[3]);
        }
        ph[0] = fmaf(tt0, tx.x, ph[0]); ph[1] = fmaf(tt0, tx.y, ph[1]);
        ph[2] = fmaf(tt0, tx.z, ph[2]); ph[3] = fmaf(tt0, tx.w, ph[3]);
        ph[0] = fmaf(tt1, ty.x, ph[0]); ph[1] = fmaf(tt1, ty.y, ph[1]);
        ph[2] = fmaf(tt1, ty.z, ph[2]); ph[3] = fmaf(tt1, ty.w, ph[3]);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) v[c] = ((mask >> (8 * c)) & 1u) ? ph[c] : 0.f;
      s1 += (v[0] + v[1]) + (v[2] + v[3]);
      if (MODE == 0) {
        s2 = fmaf(v[0], tx.x, s2); s2 = fmaf(v[1], tx.y, s2); s2 = fmaf(v[2], tx.z, s2); s2 = fmaf(v[3], tx.w, s2);
        s3 = fmaf(v[0], ty.x, s3); s3 = fmaf(v[1], ty.y, s3); s3 = fmaf(v[2], ty.z, s3); s3 = fmaf(v[3], ty.w, s3);
      } else {
        s0 += (float)__popc(mask);
        s2 = fmaf(v[0], v[0], s2); s2 = fmaf(v[1], v[1], s2); s2 = fmaf(v[2], v[2], s2); s2 = fmaf(v[3], v[3], s2);
        float rc = 0.f, rs = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f, p4 = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if ((mask >> (8 * c)) & 1u) {
            float sn, cs;
            wfm_sincos(P.k2t * v[c], sn, cs);
            rc += cs; rs += sn;
            if (MODE == 2) {
              p1 = fmaf(cs, cxw[c], p1); p2 = fmaf(sn, sxw[c], p2);
              p3 = fmaf(sn, cxw[c], p3); p4 = fmaf(cs, sxw[c], p4);
            }
          }
        }
        s3 += rc; s4 += rs;
        if (MODE == 2) {
          // row amplitudes R_a = sum_x f exp(-i a d x): a = -1: (p1 - p2, p3 + p4), 0: (rc, rs), +1: (p1 + p2, p3 - p4)
          const float sy = syw, cy = cyw;
          const float re[3] = {p1 - p2, rc, p1 + p2}, im[3] = {p3 + p4, rs, p3 - p4};
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            tc[a][0] = fmaf(re[a], cy, tc[a][0]); tc[a][1] = fmaf(im[a], sy, tc[a][1]);
            tc[a][2] = fmaf(im[a], cy, tc[a][2]); tc[a][3] = fmaf(re[a], sy, tc[a][3]);
          }
          tz[0] += re[0]; tz[1] += im[0]; tz[2] += re[2]; tz[3] += im[2];
        }
      }
    }
    if (MODE == 2) {
      const float cn = cyw * cdw - syw * sdw;
      syw = fmaf(syw, cdw, cyw * sdw);
      cyw = cn;
    }
    if (MODE == 0) *reinterpret_cast<float4*>(s_out + 20 * jl + k0) = make_float4(v[0], v[1], v[2], v[3]);
    __syncwarp();
    // the upper slot is free: fetch the screen rows of strip row i + 3 into it
    if (nl > 0 && i + 3 <= rows) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(s_up);
    }
    s_up = s_lo;
    if (++s_lo == PSW_SLOTS) { s_lo = 0; par_lo ^= 1u; }
    if (MODE == 0) {
      // lattice pass: Q[j][u] = sum_k f[16u + k] row[16j + k], one (chunk j, offset u) per lane
      const float4* q4 = reinterpret_cast<const float4*>(s_out + 20 * jl);
      float acc = 0.f;
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const float4 q = q4[k4];
        acc = fmaf(fq[4 * k4 + 0], q.x, acc); acc = fmaf(fq[4 * k4 + 1], q.y, acc);
        acc = fmaf(fq[4 * k4 + 2], q.z, acc); acc = fmaf(fq[4 * k4 + 3], q.w, acc);
      }
      s_q[lane] = acc;
      __syncwarp();
      if (lane < 11) {
        // partial T[g], g = 8 cb - 3 + lane: the chunks g + u that belong to this block
        float t = 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = lane - 3 + u;
          if (j >= 0 && j < 8) t += s_q[4 * j + u];
        }
        *tp = t;
      }
      tp += P.nb * PSW_TP;
      __syncwarp();
    }
  }

#pragma unroll
  for (int sft = 16; sft > 0; sft >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
    s1 += __shfl_xor_sync(0xffffffffu, s1, sft);
    s2 += __shfl_xor_sync(0xffffffffu, s2, sft);
    s3 += __shfl_xor_sync(0xffffffffu, s3, sft);
    s4 += __shfl_xor_sync(0xffffffffu, s4, sft);
  }
  if (lane == 0) {
    if (MODE == 0) {
      if (s1 != 0.f) atomicAdd(P.mom + (size_t)e * 4 + 0, (double)s1);
      if (s2 != 0.f) atomicAdd(P.mom + (size_t)e * 4 + 1, (double)s2);
      if (s3 != 0.f) atomicAdd(P.mom + (size_t)e * 4 + 2, (double)s3);
    } else {
      double* m = P.mom + (size_t)e * (MODE == 2 ? PSW_MOM2 : 5);
      if (s0 != 0.f) atomicAdd(m + 0, (double)s0);
      if (s1 != 0.f) atomicAdd(m + 1, (double)s1);
      if (s2 != 0.f) atomicAdd(m + 2, (double)s2);
      if (s3 != 0.f) atomicAdd(m + 3, (double)s3);
      if (s4 != 0.f) atomicAdd(m + 4, (double)s4);
    }
  }
  if (MODE == 2) {
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float t = tc[a][j];
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) t += __shfl_xor_sync(0xffffffffu, t, sft);
        if (lane == 0 && t != 0.f) atomicAdd(P.mom + (size_t)e * PSW_MOM2 + 5 + 4 * a + j, (double)t);
      }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float t = tz[j];
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) t += __shfl_xor_sync(0xffffffffu, t, sft);
      if (lane == 0 && t != 0.f) atomicAdd(P.mom + (size_t)e * PSW_MOM2 + 17 + j, (double)t);
    }
  }
}

// The nine central PSF pixels from the MODE 2 sums, normalised to a flat wavefront's peak: I[b + 1][a + 1].
__host__ __device__ inline void psw_core_pixels(const double* m, double (&I)[3][3]) {
  const double s0 = m[0], inv = s0 > 0.0 ? 1.0 / (s0 * s0) : 0.0;
  for (int a = 0; a < 3; ++a) {
    const double t1 = m[5 + 4 * a], t2 = m[6 + 4 * a], t3 = m[7 + 4 * a], t4 = m[8 + 4 * a];
    I[2][a] = ((t1 + t2) * (t1 + t2) + (t3 - t4) * (t3 - t4)) * inv;     // b = +1
    I[0][a] = ((t1 - t2) * (t1 - t2) + (t3 + t4) * (t3 + t4)) * inv;     // b = -1
  }
  I[1][0] = (m[17] * m[17] + m[18] * m[18]) * inv;
  I[1][1] = (m[3] * m[3] + m[4] * m[4]) * inv;
  I[1][2] = (m[19] * m[19] + m[20] * m[20]) * inv;
}

// Brightest of the nine pixels refined by a three-point fit per axis (a parabola through the logarithms, i.e. a Gaussian
// through the pixel and its two neighbours) when the neighbours exist inside the core; the stand-in for sutra's
// comp_strehl(do_fit=True) (un-vendored; targetCompass.py:139-196), exact same estimate as oracle/aoframe.py::psf_peak on
// the full image whenever the brightest pixel of the image is the on-axis one.
__host__ __device__ inline double psw_core_peak(const double (&I)[3][3]) {
  int bj = 1, bi = 1;
  for (int j = 0; j < 3; ++j)
    for (int i = 0; i < 3; ++i)
      if (I[j][i] > I[bj][bi]) { bj = j; bi = i; }
  const double pk = I[bj][bi];
  if (!(pk > 0.0)) return 0.0;
  double lg = log(pk);
  if (bj == 1 && I[0][bi] > 0.0 && I[2][bi] > 0.0) {
    const double m1 = log(I[0][bi]), p1 = log(I[2][bi]);
    const double a = 0.5 * (m1 + p1) - log(pk), b = 0.5 * (p1 - m1);
    if (a < 0.0) lg += -b * b / (4.0 * a);
  }
  if (bi == 1 && I[bj][0] > 0.0 && I[bj][2] > 0.0) {
    const double m1 = log(I[bj][0]), p1 = log(I[bj][2]);
    const double a = 0.5 * (m1 + p1) - log(pk), b = 0.5 * (p1 - m1);
    if (a < 0.0) lg += -b * b / (4.0 * a);
  }
  return exp(lg);
}


// Strehl figures from the MODE 2 sums: SE = fitted peak of this frame's core, LE = fitted peak of the accumulated core
// (the reference takes the maximum of the long-exposure image, not the mean of the short-exposure maxima).
// le_n / first: per-environment counts of staggered environments, as target_strehl_kernel.
__global__ void target_strehl_core_kernel(const double* mom, float* strehl, float* acc, int E, int n_le, int* le_n,
                                          const int* first) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  if (le_n) {
    if (first[e]) return;
    n_le = n_le > 0 ? ++le_n[e] : 0;
  }
  const double* m = mom + (size_t)e * PSW_MOM2;
  const double s0 = m[0];
  double I[3][3];
  psw_core_pixels(m, I);
  float var = 0.f, se = 1.f;
  if (s0 > 0.0) {
    const double mean = m[1] / s0;
    var = (float)fmax(m[2] / s0 - mean * mean, 0.0);
    se = (float)psw_core_peak(I);
  } else {
    for (int j = 0; j < 3; ++j) for (int i = 0; i < 3; ++i) I[j][i] = (j == 1 && i == 1) ? 1.0 : 0.0;
  }
  strehl[e * 4 + 0] = se;
  strehl[e * 4 + 2] = var;
  if (n_le > 0) {
    float* a = acc + (size_t)e * TAR_ACC;
    a[0] += se;
    a[1] += var;
    double L[3][3];
    for (int j = 0; j < 3; ++j)
      for (int i = 0; i < 3; ++i) {
        a[2 + 3 * j + i] += (float)I[j][i];
        L[j][i] = (double)a[2 + 3 * j + i] / (double)n_le;
      }
    strehl[e * 4 + 1] = (float)psw_core_peak(L);
    strehl[e * 4 + 3] = a[1] / (float)n_le;
  }
}
