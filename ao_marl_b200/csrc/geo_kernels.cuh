// geo_kernels.cuh -- geometric controller (ControllerType.GEO): least-squares fit of the mirrors to the turbulent
// phase of the target, com = -(IF IF^T)^-1 IF (phi - <phi>).
//
// Reference: RlSupervisor.next_part_one_geo (shesha/supervisor/rlSupervisor.py:989-1013) -> sutra's
// sutra_controller_geo (comp_dphi: phase over the pupil, average removed; comp_com: sparse IF product, then the
// dense inverse Gram matrix built by init_proj_sparse, shesha/init/rtc_init.py:418-448).  sutra's cusparse gemv over
// 1286 x 3136-pixel rows becomes two separable passes here, because every piezo row is outer(S[gy], S[gx]) of the
// shifted stamp factor:
//   geo_rows_kernel : one warp per pupil row: bilinear trace of the layers (same arithmetic as the sensor),
//                     pupil mask, row held in shared memory, T[e][y][gx] = sum_x S[gx][x] m phi(y, x);
//                     pupil sums of m phi, m phi tt_x, m phi tt_y on the side (piston term, tip-tilt rows)
//   geo_cols_kernel : b[e][a(gy,gx)] = sum_y S[gy][y] T[e][y][gx] - <phi> sum(IF_a) ; tip-tilt rows from the sums
// followed by one env-batched GEMM with -(IF IF^T)^+ (AOM_T_GEO_PROJ).  The phase is never materialised; T is
// [E][n][gp] floats (gp = lattice side rounded to 16), 8 % of a pupil-plane cube.
// On the production lattices (pitch 16) the row pass is MODE 0 of pupil_sweep.cuh (staged screen rows, vector loads);
// geo_rows_kernel below is the generic form for any pitch.
#pragma once
#include "wfs_kernels.cuh"

#define GEO_ROW_WARPS 4

template <bool PE = false>      // PE: per-environment winds (layer offsets from p.wind)
__global__ void __launch_bounds__(GEO_ROW_WARPS * 32) geo_rows_kernel(WfsParams p, float* __restrict__ T, int gp,
                                                                       double* __restrict__ mom) {
  extern __shared__ float s_rows[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.y, y = blockIdx.x * GEO_ROW_WARPS + warp;
  if (y >= p.n) return;                      // whole warp
  const int rs = p.n + (p.n >> 4) + 2;       // pixel x sits at x + (x >> 4): lattice columns 16 px apart hit 17 banks
  float* row = s_rows + warp * rs;
  float s1 = 0.f, sx = 0.f, sy = 0.f;
  const float* mrow = p.mpupil + (size_t)y * p.n;
  const float* ttx = p.tt_planes + (size_t)(y + p.tt_off) * p.tt_dim + p.tt_off;
  const float* tty = ttx + (size_t)p.tt_dim * p.tt_dim;
  for (int x = lane; x < p.n; x += 32) {
    float v = 0.f;
    if (mrow[x] != 0.f) {
      for (int l = 0; l < p.n_layers; ++l) {
        const WfsLayer& L = p.layer[l];
        const int N = L.N;
        const float* scr = L.screen + (size_t)e * N * N;
        const int ox = L.ox[e], oy = L.oy[e];
        const WindRec w = wind_of<PE>(p, l, e);
        // footprint inside the screen (checked on the host) and 0 <= ox, oy < N: one conditional subtract wraps
        int pc0 = x + w.ix + ox; pc0 -= (pc0 >= N) ? N : 0;
        int pc1 = pc0 + 1;       pc1 -= (pc1 >= N) ? N : 0;
        int pr0 = y + w.iy + oy; pr0 -= (pr0 >= N) ? N : 0;
        int pr1 = pr0 + 1;       pr1 -= (pr1 >= N) ? N : 0;
        float top = wfs_layer_row(scr, N, pr0, pc0, pc1, w.fx);
        float bot = wfs_layer_row(scr, N, pr1, pc0, pc1, w.fx);
        v += top + w.fy * (bot - top);
      }
      s1 += v;
      sx = fmaf(v, __ldg(ttx + x), sx);
      sy = fmaf(v, __ldg(tty + x), sy);
    }
    row[x + (x >> 4)] = v;
  }
  __syncwarp();
  for (int g = lane; g < p.grid_n; g += 32) {
    const int xs = p.i1_0 + g * p.pitch - p.pzt_off;
    const int d0 = max(0, -xs), d1 = min(p.ss, p.n - xs);
    float t = 0.f;
    for (int d = d0; d < d1; ++d) {
      const int x = xs + d;
      t = fmaf(__ldg(p.stamp1d + d), row[x + (x >> 4)], t);
    }
    T[((size_t)e * p.n + y) * gp + g] = t;
  }
#pragma unroll
  for (int sft = 16; sft > 0; sft >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, sft);
    sx += __shfl_xor_sync(0xffffffffu, sx, sft);
    sy += __shfl_xor_sync(0xffffffffu, sy, sft);
  }
  if (lane == 0 && (s1 != 0.f || sx != 0.f || sy != 0.f)) {
    atomicAdd(mom + (size_t)e * 4 + 0, (double)s1);
    atomicAdd(mom + (size_t)e * 4 + 1, (double)sx);
    atomicAdd(mom + (size_t)e * 4 + 2, (double)sy);
  }
}

// sifn [nactu]: pupil sum of each influence row divided by the number of pupil points.
// nb == 0: T is [E][n][gp] (geo_rows_kernel); nb > 0: T holds the sweep's per-block partial sums [E][n][nb][12], entry
// t of block cb = lattice column 8 cb - 3 + t restricted to the block's chunks (pupil_sweep.cuh): a column's own
// block and, when its stamp reaches into the next one ((gx & 7) >= 5), that one too.
__global__ void geo_cols_kernel(WfsParams p, const float* __restrict__ T, int gp, int nb, const double* __restrict__ mom,
                                const float* __restrict__ sifn, float* __restrict__ bvec, int ldb) {
  const int e = blockIdx.x;
  const double s1 = mom[(size_t)e * 4];
  const float s1f = (float)s1;
  const int rowf = nb > 0 ? nb * 12 : gp;
  const float* Te = T + (size_t)e * p.n * rowf;
  const int cells = p.grid_n * p.grid_n;
  for (int c = threadIdx.x; c < cells; c += blockDim.x) {
    const int a = p.act_map[c];
    if (a < 0) continue;
    const int gy = c / p.grid_n, gx = c - gy * p.grid_n;
    const int ys = p.j1_0 + gy * p.pitch - p.pzt_off;
    const int d0 = max(0, -ys), d1 = min(p.ss, p.n - ys);
    float t = 0.f;
    if (nb > 0) {
      const int cb = gx >> 3;
      const int o0 = cb * 12 + (gx & 7) + 3;
      const bool two = (gx & 7) >= 5 && cb + 1 < nb;
      const int o1 = (cb + 1) * 12 + (gx & 7) - 5;
      for (int d = d0; d < d1; ++d) {
        const float* r = Te + (size_t)(ys + d) * rowf;
        float v = r[o0];
        if (two) v += r[o1];
        t = fmaf(__ldg(p.stamp1d + d), v, t);
      }
    } else {
      for (int d = d0; d < d1; ++d) t = fmaf(__ldg(p.stamp1d + d), Te[(size_t)(ys + d) * gp + gx], t);
    }
    bvec[(size_t)e * ldb + a] = t - s1f * sifn[a];
  }
  if (threadIdx.x < 2) {
    const int a = p.pzt_nact + threadIdx.x;
    bvec[(size_t)e * ldb + a] = (float)(mom[(size_t)e * 4 + 1 + threadIdx.x] - s1 * (double)sifn[a]);
  }
}
