// Turbulence screens: ring-buffered storage + batched extrusion.
//
// Reference maths: shesha/util/iterkolmo.py:255-288 (extrude), scheduling in sutra's Atmos.move_atmos
// behind shesha/supervisor/components/atmosCompass.py:158-161.  The reference shifts the whole
// N x N screen by one pixel per extrusion (read + write of 1.7 MB per layer); here every screen is a
// torus addressed through per-environment offsets (ox, oy):
//        logical (y, x)  ->  physical ((y + oy) mod N, (x + ox) mod N)
// so an extrusion only writes the N new pixels.  The four directions reuse the single +x stencil:
//        +x: (r, c)          -x: (N-1-r, N-1-c)        (iterkolmo.py:246-249 mirror)
//        +y: (c, r)          -y: (N-1-c, N-1-r)        (iterkolmo.py:241-244 transpose)
// One extrusion of all E environments = gather Z [E][S+N] -> GEMM with [A|B] -> scatter N pixels.
#pragma once
#include <cuda_runtime.h>
#include "../../include/aomarl.h"
#include "rng.cuh"
#include "wind_host.h"

struct ExtrudeParams {
  float* screen;          // [E][N][N]
  int* ox; int* oy;       // [E]
  uint32_t* count;        // [E] extrusions done since reset (RNG counter)
  const uint32_t* k0; const uint32_t* k1;   // [E] Philox key = env seed
  const int* stencil;     // [S]
  float* Z; int ldz;      // [E][ldz]
  float* zref;            // [E]
  float* newcol; int ldn; // [E][ldn]
  int N, S, E, layer, axis, sign;
  float amp;
  const float* amp_env;   // [E] per-environment amplitude, or null
  // per-environment winds (the PE instantiations): signed whole-pixel counts of this axis for this frame [E]; pass
  // `pass` extrudes environment e iff pass < |steps[e]|, with the sign of steps[e] (`sign` is not read).  An environment
  // that sits out a pass is not touched: no gather, no store, no RNG counter increment.
  const int* steps;
  int pass;
  // compacted start-up (aom_reset_envs): row k of Z / zref / newcol belongs to environment envs[k]; null: row e = environment e
  const int* envs;
};

// the direction of this pass for environment e; false: e sits it out
template <bool PE>
__device__ __forceinline__ bool extr_active(const int* steps, int pass, int e, int& sign) {
  if (!PE) return true;
  const int n = steps[e];
  sign = n < 0 ? -1 : 1;
  return pass < (n < 0 ? -n : n);
}

__device__ __forceinline__ void extr_logical(int r, int c, int N, int axis, int sign, int& lr, int& lc) {
  if (axis == 0) { lr = r; lc = c; } else { lr = c; lc = r; }
  if (sign < 0) {
    if (axis == 0) { lr = N - 1 - r; lc = N - 1 - c; } else { lr = N - 1 - c; lc = N - 1 - r; }
  }
}

__device__ __forceinline__ int wrapN(int v, int N) { return v >= N ? v - N : v; }

// grid: E blocks of 256 threads.  One block walks the whole input vector of its environment: the per-element
// dependent chain (stencil index -> screen pixel) is pipelined over ~5 iterations per thread instead of being paid
// once per 256-thread block (32 k tiny blocks per launch were block-latency bound: 75 us per launch), and one
// Philox block yields its four innovations instead of one.
template <bool PE = false>
__global__ void __launch_bounds__(256) extrude_gather_kernel(ExtrudeParams p) {
  const int row = blockIdx.x, e = p.envs ? p.envs[row] : row;
  int sign = p.sign;
  if (!extr_active<PE>(p.steps, p.pass, e, sign)) return;
  const int N = p.N;
  const float* scr = p.screen + (size_t)e * N * N;
  const int ox = p.ox[e], oy = p.oy[e];
  // reference pixel: p'[0, N-1] of the rotated/transposed screen
  int rr, rc;
  extr_logical(0, N - 1, N, p.axis, sign, rr, rc);
  const float zr = scr[(size_t)wrapN(rr + oy, N) * N + wrapN(rc + ox, N)];
  if (threadIdx.x == 0) p.zref[row] = zr;
  float* Z = p.Z + (size_t)row * p.ldz;
  for (int k = threadIdx.x; k < p.S; k += blockDim.x) {
    const int idx = p.stencil[k];
    int lr, lc;
    extr_logical(idx / N, idx % N, N, p.axis, sign, lr, lc);
    Z[k] = scr[(size_t)wrapN(lr + oy, N) * N + wrapN(lc + ox, N)] - zr;
  }
  const uint32_t cnt = p.count[e], k0 = p.k0[e], k1 = p.k1[e];
  const float amp = p.amp_env ? p.amp_env[e] : p.amp;
  for (int b = threadIdx.x; 4 * b < N; b += blockDim.x) {
    const aom_u4 w = aom_philox((uint32_t)b, cnt, AOM_TAG_ATMOS, (uint32_t)p.layer, k0, k1);
    float z[4];
    aom_normal_pair(w.x, w.y, z[0], z[1]);
    aom_normal_pair(w.z, w.w, z[2], z[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (4 * b + i < N) Z[p.S + 4 * b + i] = aom_mul(z[i], amp);
  }
  for (int k = p.S + N + threadIdx.x; k < p.ldz; k += blockDim.x) Z[k] = 0.f;
}

// grid: E (or K compacted) blocks of EXTRUDE_SCATTER_THREADS threads, one block per environment, every thread holds its (up to 8) pixels
// of the new column in registers before it stores them.  A row-direction extrusion (contiguous) takes 9 us per 4096
// environments (15 us with one warp per environment and a load -> store loop).  A column-direction extrusion is 648
// four-byte stores into 648 different DRAM rows per environment -- a read-modify-write of a sector each, 91 MB read +
// 81 MB written for 10.6 MB of pixels -- and stays at 117 us however many stores are in flight (120 us before): it is
// bound by DRAM row activations (profiles/r02_extrude_kernels_metrics.csv), the price of storing every layer [y][x].
#define EXTRUDE_SCATTER_THREADS 128
template <bool PE = false>
__global__ void __launch_bounds__(EXTRUDE_SCATTER_THREADS) extrude_scatter_kernel(ExtrudeParams p) {
  const int row = blockIdx.x, e = p.envs ? p.envs[row] : row;
  int sign = p.sign;
  if (!extr_active<PE>(p.steps, p.pass, e, sign)) return;
  const int N = p.N;
  float* scr = p.screen + (size_t)e * N * N;
  const int ox = p.ox[e], oy = p.oy[e];
  const float zr = p.zref ? p.zref[row] : 0.f;         // null: the GEMM already added the reference pixel
  int nox = ox, noy = oy;
  if (p.axis == 0) nox = (sign > 0) ? wrapN(ox + 1, N) : (ox == 0 ? N - 1 : ox - 1);
  else             noy = (sign > 0) ? wrapN(oy + 1, N) : (oy == 0 ? N - 1 : oy - 1);
  const float* col = p.newcol + (size_t)row * p.ldn;
  constexpr int PER = 8;                                    // pixels per thread and pass (N <= 1024 in one pass)
  for (int j0 = threadIdx.x; j0 < N; j0 += PER * EXTRUDE_SCATTER_THREADS) {
    float v[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int j = j0 + i * EXTRUDE_SCATTER_THREADS;
      v[i] = (j < N) ? col[j] + zr : 0.f;
    }
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int j = j0 + i * EXTRUDE_SCATTER_THREADS;
      if (j < N) {
        size_t addr;
        if (p.axis == 0) {
          const int pc = (sign > 0) ? ox : nox;                 // new logical column N-1 (or 0)
          const int lr = (sign > 0) ? j : N - 1 - j;
          addr = (size_t)wrapN(lr + oy, N) * N + pc;
        } else {
          const int pr = (sign > 0) ? oy : noy;                 // new logical row N-1 (or 0)
          const int lc = (sign > 0) ? j : N - 1 - j;
          addr = (size_t)pr * N + wrapN(lc + ox, N);
        }
        scr[addr] = v[i];
      }
    }
  }
  __syncthreads();                                            // every thread has read the old ring origin
  if (threadIdx.x == 0) {
    p.ox[e] = nox;
    p.oy[e] = noy;
    p.count[e] += 1;
  }
}

// In-place transpose of E square screens [N][N].  grid (T (T + 1) / 2, E) with T = ceil(N / 32): every block swaps one pair
// of 32 x 32 tiles (bi <= bj) through shared memory; block (32, 8).  Used by the start-up of aom_reset / aom_reset_envs,
// which runs its 2N extrusions along the contiguous axis of a transposed screen (see there).  envs: grid.y = K and
// block row k transposes the screen of environment envs[k]; null: environment blockIdx.y.
__global__ void __launch_bounds__(256) transpose_screens_kernel(float* __restrict__ screens, int N, const int* __restrict__ envs) {
  __shared__ float ta[32][33], tb[32][33];
  const int T = (N + 31) / 32;
  // tile pair index -> (bi, bj), bi <= bj
  int t = blockIdx.x, bi = 0;
  while (t >= T - bi) { t -= T - bi; ++bi; }
  const int bj = bi + t;
  float* scr = screens + (size_t)(envs ? envs[blockIdx.y] : (int)blockIdx.y) * N * N;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int r = ty; r < 32; r += 8) {
    const int ya = bi * 32 + r, xa = bj * 32 + tx;            // tile A = (rows of bi, columns of bj)
    ta[r][tx] = (ya < N && xa < N) ? scr[(size_t)ya * N + xa] : 0.f;
    const int yb = bj * 32 + r, xb = bi * 32 + tx;            // tile B = (rows of bj, columns of bi)
    tb[r][tx] = (yb < N && xb < N) ? scr[(size_t)yb * N + xb] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int ya = bi * 32 + r, xa = bj * 32 + tx;
    if (ya < N && xa < N) scr[(size_t)ya * N + xa] = tb[tx][r];   // A <- B^T
    const int yb = bj * 32 + r, xb = bi * 32 + tx;
    if (bi != bj && yb < N && xb < N) scr[(size_t)yb * N + xb] = ta[tx][r];   // B <- A^T
  }
}

// Wind state of every layer and environment when the environments have their own winds: accumulators acc [L][2][E]
// (x, y), whole-pixel counts of the frame steps [L][2][E] (x, y) and the samplers' offsets rec [L][E].  One thread per
// (layer, environment), the arithmetic of wind_host.h (the host keeps a mirror of the accumulators with the same
// functions, wind_mirror, to know how many extrusion passes to launch).  The modes are those of wind_host.h.
struct WindStateParams {
  WindLayerParams layer[AOM_MAX_LAYERS];
  double* acc; int* steps; WindRec* rec;
  int E, n_layers, mode;
  const int* envs; int K;                // WIND_RESET_ENVS
};

// grid: one thread per (layer, environment), or per (layer, listed environment) with WIND_RESET_ENVS.
__global__ void wind_state_kernel(const __grid_constant__ WindStateParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = P.mode == WIND_RESET_ENVS ? P.K : P.E;
  if (i >= P.n_layers * n) return;
  const int l = i / n, k = i - l * n;
  const int e = P.mode == WIND_RESET_ENVS ? P.envs[k] : k;
  const WindLayerParams& L = P.layer[l];
  const float dx = L.dx ? L.dx[e] : L.cdx, dy = L.dy ? L.dy[e] : L.cdy;
  double* ax = P.acc + (size_t)2 * l * P.E + e;
  double* ay = ax + P.E;
  double x = 0.0, y = 0.0;
  int nx = 0, ny = 0;
  if (P.mode == WIND_STEP) {
    x = *ax; y = *ay;
    nx = wind_advance(x, dx);
    ny = wind_advance(y, dy);
  } else if (P.mode == WIND_INIT) {
    x = L.ax0; y = L.ay0;
  } else {
    ny = dx < 0.f ? -L.n2 : L.n2;
  }
  *ax = x; *ay = y;
  P.steps[(size_t)2 * l * P.E + e] = nx;
  P.steps[(size_t)(2 * l + 1) * P.E + e] = ny;
  P.rec[(size_t)l * P.E + e] = wind_record(L.xoff, L.yoff, x, y);
}

// WIND_LOAD_ENVS (aom_load_envs): accumulators of the listed environments envs[0..K) <- acc_in [L][2][K], no extrusion.
// One thread per (layer, listed environment); the others keep their state.
struct WindLoadParams {
  float xoff[AOM_MAX_LAYERS], yoff[AOM_MAX_LAYERS];
  double* acc; int* steps; WindRec* rec;
  const int* envs; const double* acc_in;
  int E, K, n_layers;
};

__global__ void wind_load_kernel(const __grid_constant__ WindLoadParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n_layers * P.K) return;
  const int l = i / P.K, k = i - l * P.K, e = P.envs[k];
  const double x = P.acc_in[(size_t)2 * l * P.K + k], y = P.acc_in[(size_t)(2 * l + 1) * P.K + k];
  P.acc[(size_t)2 * l * P.E + e] = x;
  P.acc[(size_t)(2 * l + 1) * P.E + e] = y;
  P.steps[(size_t)2 * l * P.E + e] = 0;
  P.steps[(size_t)(2 * l + 1) * P.E + e] = 0;
  P.rec[(size_t)l * P.E + e] = wind_record(P.xoff[l], P.yoff[l], x, y);
}
