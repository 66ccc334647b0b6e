// FP32 GEMM for the env-batched contractions of the step (screen extrusion, command-matrix
// reconstruction, Btt projections, actor layers):
//
//        C[b][m][n] = sum_k A[b][m][k] * B[b][n][k]  (+ bias[b][n]) (relu)        "TN", both K-major
//
// A = per-environment vectors [E][ld], B = shared operator [rows][ld]; leading dimensions are
// multiples of 16 floats and pad columns hold zeros, so K is walked in whole 16-wide slabs with
// aligned 128-bit loads and no K predicate.  128 x 128 x 16 tiles, 256 threads, 8 x 8 register
// blocking, register-staged double buffering.  Round-1 SIMT kernel: exact fp32 accumulation so that
// commands / rewards stay within rel 1e-4 of the oracle; the tcgen05 (3xTF32) version replaces it.
#pragma once
#include <cuda_runtime.h>

#define GEMM_BM 128
#define GEMM_BN 128
#define GEMM_BK 16
#define GEMM_PAD 4

struct GemmParams {
  const float* A; const float* B; float* C; const float* bias;
  int lda, ldb, ldc;
  int M, N, K;          // K rounded up to a multiple of 16 by the caller (operands are zero padded)
  long long sA, sB, sC, sBias;   // batch strides (elements)
  int relu;
  // epilogue 1 (integrator): err = -acc ; C = err ; com += gain * err
  float* com; int ldcom; float gain; int closed;
  // gemm_tc_kernel only: the B operand already split into TF32 hi / lo planes in the UMMA tile order of 128-column tiles
  // ([n tile][k block][hi, lo][128 x 16]; gtc_pretile_host), brought in by one bulk copy per stage.  Null: B is split on the fly.
  const float* Bt; long long sBt;
  // epilogue 2: the integrator of epilogue 1 with one gain per row (environment): com += gain_env[row] * err
  const float* gain_env;
};

template <int EPI>
__global__ void __launch_bounds__(256, 2) gemm_tn_kernel(GemmParams p) {
  __shared__ __align__(16) float As[2][GEMM_BK][GEMM_BM + GEMM_PAD];
  __shared__ __align__(16) float Bs[2][GEMM_BK][GEMM_BN + GEMM_PAD];
  const int tid = threadIdx.x;
  const int bz = blockIdx.z;
  const float* __restrict__ A = p.A + (long long)bz * p.sA;
  const float* __restrict__ B = p.B + (long long)bz * p.sB;
  float* __restrict__ C = p.C + (long long)bz * p.sC;
  const int m0 = blockIdx.y * GEMM_BM;
  const int n0 = blockIdx.x * GEMM_BN;

  // global -> smem staging: each thread moves two float4 of A and two of B per slab
  const int lrow = tid >> 2;          // 0..63
  const int lk = (tid & 3) << 2;      // 0,4,8,12
  float4 ra[2], rb[2];
  auto load_slab = [&](int k0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int row = m0 + lrow + h * 64;
      ra[h] = (row < p.M) ? *reinterpret_cast<const float4*>(A + (long long)row * p.lda + k0 + lk)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
      int col = n0 + lrow + h * 64;
      rb[h] = (col < p.N) ? *reinterpret_cast<const float4*>(B + (long long)col * p.ldb + k0 + lk)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto store_slab = [&](int buf) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int r = lrow + h * 64;
      As[buf][lk + 0][r] = ra[h].x; As[buf][lk + 1][r] = ra[h].y;
      As[buf][lk + 2][r] = ra[h].z; As[buf][lk + 3][r] = ra[h].w;
      Bs[buf][lk + 0][r] = rb[h].x; Bs[buf][lk + 1][r] = rb[h].y;
      Bs[buf][lk + 2][r] = rb[h].z; Bs[buf][lk + 3][r] = rb[h].w;
    }
  };

  const int ty = tid >> 4;   // 0..15 -> rows ty*4 .. +4 and 64 + ty*4 .. +4
  const int tx = tid & 15;   // 0..15 -> cols tx*4 .. +4 and 64 + tx*4 .. +4
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int nslab = p.K / GEMM_BK;
  load_slab(0);
  store_slab(0);
  __syncthreads();
  for (int s = 0; s < nslab; ++s) {
    const int buf = s & 1;
    if (s + 1 < nslab) load_slab((s + 1) * GEMM_BK);
#pragma unroll
    for (int k = 0; k < GEMM_BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
      float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (s + 1 < nslab) {
      store_slab(buf ^ 1);
      __syncthreads();
    }
  }

  const float* bias = p.bias ? p.bias + (long long)bz * p.sBias : nullptr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (row >= p.M) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      int col = n0 + jh * 64 + tx * 4;
      if (col >= p.ldc) continue;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int c = col + j;
        float x = acc[i][jh * 4 + j];
        if (EPI == 0) {
          if (bias && c < p.N) x += bias[c];
          if (p.relu) x = fmaxf(x, 0.f);
        } else {
          x = -x;
        }
        v[j] = (c < p.N) ? x : 0.f;   // pad columns stay zero
      }
      *reinterpret_cast<float4*>(C + (long long)row * p.ldc + col) = make_float4(v[0], v[1], v[2], v[3]);
      if ((EPI == 1 || EPI == 2) && p.closed) {
        const float g = (EPI == 2) ? p.gain_env[row] : p.gain;
        float4* cp = reinterpret_cast<float4*>(p.com + (long long)row * p.ldcom + col);
        float4 c4 = *cp;
        c4.x = fmaf(g, v[0], c4.x); c4.y = fmaf(g, v[1], c4.y);
        c4.z = fmaf(g, v[2], c4.z); c4.w = fmaf(g, v[3], c4.w);
        *cp = c4;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Exact-fp32 GEMM for the screen extrusion, shaped to the operator: C[M][N] = A[M][K] . B[N][K]^T with
// round-to-nearest FFMA accumulation (the autoregressive screens integrate the ~1e-5 shrink a truncating
// tensor-core accumulator would add, DESIGN.md section 4).  N is the screen side (648 / 168), which the square
// 128 x 128 tiles of gemm_tn_kernel quantise badly (6 column tiles for 5.06, 192 CTAs on 296 slots).  Here a CTA
// of 128 threads owns a 128 x (8 CN) tile, CN = 9 -> 72 columns -> 9 x 32 = 288 CTAs for N = 648, M = 4096: one
// full wave at two CTAs per SM and no padded columns.  Thread (ty, tx) = (tid / 8, tid % 8) accumulates rows
// 8 ty .. 8 ty + 7 x columns CN tx .. CN tx + CN - 1: 8 x CN independent FFMA chains fed by 2 LDS.128 + CN
// conflict-free LDS.32 per k (row stride BN + 1).  Measured on B200, N = 648, M = 4096: 0.315 ms per extrusion
// against 0.42 ms for the square tiles; splitting the column reads into LDS.128 groups was slower (0.34 ms).
template <int CN>
__global__ void __launch_bounds__(128, 4) gemm_tn_exact_kernel(GemmParams p) {
  constexpr int BN = 8 * CN;
  constexpr int BPAD = 1;       // row stride BN + 1: the CN-strided column reads of a warp hit distinct banks
  static_assert(CN == 8 || CN == 9, "column tile is 64 or 72 wide");
  __shared__ __align__(16) float As[2][GEMM_BK][GEMM_BM + GEMM_PAD];
  __shared__ __align__(16) float Bs[2][GEMM_BK][BN + BPAD];
  const int tid = threadIdx.x;
  const float* __restrict__ A = p.A;
  const float* __restrict__ B = p.B;
  float* __restrict__ C = p.C;
  const int m0 = blockIdx.y * GEMM_BM;
  const int n0 = blockIdx.x * BN;

  // staging: A slab = 128 rows x 4 float4 -> 4 per thread; B slab = BN rows x 4 float4 -> up to 3 per thread
  constexpr int B_ITERS = (BN * 4 + 127) / 128;
  const int lk = (tid & 3) << 2;
  const int lrow = tid >> 2;            // 0..31
  float4 ra[4], rb[B_ITERS];
  auto load_slab = [&](int k0) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const int row = m0 + lrow + h * 32;
      ra[h] = (row < p.M) ? *reinterpret_cast<const float4*>(A + (long long)row * p.lda + k0 + lk)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int h = 0; h < B_ITERS; ++h) {
      const int r = lrow + h * 32, col = n0 + r;
      rb[h] = (r < BN && col < p.N) ? *reinterpret_cast<const float4*>(B + (long long)col * p.ldb + k0 + lk)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto store_slab = [&](int buf) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const int r = lrow + h * 32;
      As[buf][lk + 0][r] = ra[h].x; As[buf][lk + 1][r] = ra[h].y;
      As[buf][lk + 2][r] = ra[h].z; As[buf][lk + 3][r] = ra[h].w;
    }
#pragma unroll
    for (int h = 0; h < B_ITERS; ++h) {
      const int r = lrow + h * 32;
      if (r < BN) {
        Bs[buf][lk + 0][r] = rb[h].x; Bs[buf][lk + 1][r] = rb[h].y;
        Bs[buf][lk + 2][r] = rb[h].z; Bs[buf][lk + 3][r] = rb[h].w;
      }
    }
  };

  const int ty = tid >> 3, tx = tid & 7;
  float acc[8][CN];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < CN; ++j) acc[i][j] = 0.f;

  // split K over gridDim.z CTAs (partial sums are added with red.global.add onto a zeroed C: two round-to-nearest
  // partial sums, commutative, so the result stays deterministic and unbiased)
  const int nslab_all = p.K / GEMM_BK;
  const int per = (nslab_all + gridDim.z - 1) / gridDim.z;
  const int slab0 = blockIdx.z * per;
  const int nslab = min(per, nslab_all - slab0);
  if (nslab <= 0) return;
  load_slab(slab0 * GEMM_BK);
  store_slab(0);
  __syncthreads();
  for (int s = 0; s < nslab; ++s) {
    const int buf = s & 1;
    if (s + 1 < nslab) load_slab((slab0 + s + 1) * GEMM_BK);
#pragma unroll
    for (int k = 0; k < GEMM_BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8 + 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[CN];
#pragma unroll
      for (int j = 0; j < CN; ++j) bv[j] = Bs[buf][k][tx * CN + j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < CN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (s + 1 < nslab) {
      store_slab(buf ^ 1);
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + ty * 8 + i;
    if (row >= p.M) continue;
#pragma unroll
    for (int j = 0; j < CN; ++j) {
      const int c = n0 + tx * CN + j;
      if (gridDim.z > 1) {
        if (c < p.N) atomicAdd(C + (long long)row * p.ldc + c, acc[i][j]);
      } else if (c < p.ldc) {
        C[(long long)row * p.ldc + c] = (c < p.N) ? acc[i][j] : 0.f;   // pad columns stay zero
      }
    }
  }
}
