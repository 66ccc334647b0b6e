// Digit code of the exact integer contraction (extrude_i8.cuh): tile geometry, row exponents, signed 7-bit digits and the
// host slicing of an operator.  Plain C++ without the CUDA headers, so that the CPU test harness
// (tests/cpu_kernels/harness.cpp) checks the same code the library runs at aom_set_table and in its kernels.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define OZ_HD __host__ __device__ __forceinline__
#else
#define OZ_HD inline
#endif

#define OZ_SLICES 6                               // digits of the per-extrusion inputs (41 bits below the row maximum)
#define OZ_SLICES_B 6                             // digits of the operator rows (41 bits): its truncation is a FIXED perturbation
                                                  // of the recursion and adds up coherently -- with 4 digits the 648^2 screens
                                                  // were 9.5e-5 off after a reset (measured, and reproduced in numpy)
#define OZ_LEVELS 6                               // digit pairs kept: s + t <= 5
#define OZ_LEVELS_PRODUCT 5                       // controller products (no recursion behind them): s + t <= 4, 15 MMAs per k
                                                  // block (with s + t <= 3 the 40x40 closed loop moved from 1e-6 to 1e-5 .. 4e-5
                                                  // of the oracle: measured, profiles/r02_parity_levels4.json)
#define OZ_BM 128
#define OZ_BN 80
#define OZ_BK 32
#define OZ_A_TILE (OZ_BM * OZ_BK)                 // 4096 bytes: one digit plane of 128 rows x 32 k
#define OZ_B_TILE (OZ_BN * OZ_BK)                 // 2560 bytes
#define OZ_EV_NONFINITE 0x40000000                // row exponent of an input row holding a NaN or an infinity: every output
                                                  // of the row is NaN

// element (row r, k) of a [rows x 32] int8 tile: 8-row x 16-byte core matrices, 128 B between the two k halves,
// 256 B between 8-row groups
OZ_HD uint32_t oz_tile_offset(int r, int kk) {
  return (uint32_t)((r >> 3) * 256 + (kk >> 4) * 128 + (r & 7) * 16 + (kk & 15));
}

// NS signed 7-bit digits of x * scale, |x * scale| < 1 (every step is exact in float64 for inputs of <= 48 bits)
template <int NS>
OZ_HD void oz_digits(double x, double scale, int (&q)[NS]) {
  double t = x * scale * 64.0;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const double r = rint(t);
    q[s] = (int)r;
    t = (t - r) * 128.0;
  }
}

// the same digits of a float32 value: every step is exact in float32 (the remainders only lose leading bits)
template <int NS>
OZ_HD void oz_digits_f32(float x, float scale, int (&q)[NS]) {
  float t = x * scale * 64.0f;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const float r = rintf(t);
    q[s] = (int)r;
    t = (t - r) * 128.0f;
  }
}

// power of two e with |x| * 2^-e in [0.5, 1) for the row maximum x (0 for an all-zero row)
OZ_HD int oz_exponent(double amax) {
  if (!(amax > 0.0)) return 0;
  int e;
  frexp(amax, &e);           // amax = m 2^e, m in [0.5, 1)
  return e;
}

// Host: nonzero when the K valid columns of every one of the `rows` rows of the operator [rows][ld] are finite
static inline int oz_operator_finite(const float* AB, int rows, int ld, int K) {
  for (int n = 0; n < rows; ++n)
    for (int k = 0; k < K; ++k)
      if (!isfinite(AB[(size_t)n * ld + k])) return 0;
  return 1;
}

// Host: cut the rows of the finite operator [rows][ld] (K valid columns) into digit planes in the tile layout of the kernel:
// [NT][KB][OZ_SLICES_B][OZ_B_TILE].  planes: NT * KB * OZ_SLICES_B * OZ_B_TILE bytes (zero-initialised by the caller);
// ea: NT * OZ_BN ints (0 for the pad rows).
static inline void oz_slice_operator(const float* AB, int rows, int ld, int K, int KB, int NT, uint8_t* planes, int* ea) {
  for (int n = 0; n < NT * OZ_BN; ++n) {
    ea[n] = 0;
    if (n >= rows) continue;
    const float* row = AB + (size_t)n * ld;
    double amax = 0.0;
    for (int k = 0; k < K; ++k) amax = fmax(amax, fabs((double)row[k]));
    const int ex = oz_exponent(amax);
    ea[n] = ex;
    const double scale = ldexp(1.0, -ex);
    const int nt = n / OZ_BN, r = n % OZ_BN;
    for (int k = 0; k < K; ++k) {
      int q[OZ_SLICES_B];
      oz_digits<OZ_SLICES_B>((double)row[k], scale, q);
      const int kb = k / OZ_BK, kk = k % OZ_BK;
      for (int s = 0; s < OZ_SLICES_B; ++s)
        planes[((size_t)(nt * KB + kb) * OZ_SLICES_B + s) * OZ_B_TILE + oz_tile_offset(r, kk)] = (uint8_t)(int8_t)q[s];
    }
  }
}
