// Host build of the device math headers (rng.cuh, fft16.cuh) and of the host-only headers the library prepares its kernels
// with (gemm_tc_host.h, wfs_lattice_host.h, extrude_i8_digits.h), so that the exact code the library runs can be checked against the numpy
// oracle on a machine without a GPU.
// Built by tests/test_cpu_kernels.py:  g++ -O2 -ffp-contract=off -shared -fPIC
#include <cmath>
#include <cstdint>
#include <vector>
#include "../../ao_marl_b200/csrc/rng.cuh"
#include "../../ao_marl_b200/csrc/fft16.cuh"
#include "../../ao_marl_b200/csrc/gemm_tc_host.h"
#include "../../ao_marl_b200/csrc/wfs_lattice_host.h"
#include "../../ao_marl_b200/csrc/extrude_i8_digits.h"

extern "C" {

void h_philox(int n, const uint32_t* c0, const uint32_t* c1, const uint32_t* c2, const uint32_t* c3,
              uint32_t k0, uint32_t k1, uint32_t* out) {
  for (int i = 0; i < n; ++i) {
    aom_u4 w = aom_philox(c0[i], c1[i], c2[i], c3[i], k0, k1);
    out[4 * i] = w.x; out[4 * i + 1] = w.y; out[4 * i + 2] = w.z; out[4 * i + 3] = w.w;
  }
}

void h_det(int n, const float* x, float* lg, float* ex, float* c, float* s) {
  for (int i = 0; i < n; ++i) {
    lg[i] = aom_det_log(x[i]);
    ex[i] = aom_det_exp(-30.0f * x[i]);
    aom_det_sincos2pi(x[i], c[i], s[i]);
  }
}

// n normals of stream (tag, sub) at counter word n_ctr, key = seed
void h_normals(int n, int64_t seed, uint32_t n_ctr, uint32_t tag, uint32_t sub, float* out) {
  uint32_t k0 = (uint32_t)((uint64_t)seed & 0xffffffffu), k1 = (uint32_t)((uint64_t)seed >> 32);
  for (int j = 0; j < n; ++j) {
    aom_u4 w = aom_philox((uint32_t)(j >> 2), n_ctr, tag, sub, k0, k1);
    out[j] = aom_normal_of_block(w, j & 3);
  }
}

void h_pixel_noise(int n, const float* lam, float noise, int64_t seed, uint32_t frame, uint32_t wfs, float* out) {
  uint32_t k0 = (uint32_t)((uint64_t)seed & 0xffffffffu), k1 = (uint32_t)((uint64_t)seed >> 32);
  for (int i = 0; i < n; ++i) out[i] = aom_pixel_noise(lam[i], noise, (uint32_t)i, frame, wfs, k0, k1);
}

// raw Poisson sampler on explicit Philox words (tail known-answer tests)
void h_poisson(int n, const float* lam, const uint32_t* x0, const uint32_t* x1, int32_t* out) {
  for (int i = 0; i < n; ++i) out[i] = aom_poisson(lam[i], x0[i], x1[i]);
}

// Pruned 2-D spot: in [16][16] complex -> intensity on the centred (2H x 2H) grid, H = 4R,
// computed exactly as the kernel does (rows then columns, one aom_fft16_pruned per (vector, b)).
void h_spot(int R, const float* inr, const float* ini, float* inten) {
  const int N = 16 * R, H = 4 * R, W = 2 * H;
  std::vector<float> twr(R * 16), twi(R * 16);
  for (int b = 0; b < R; ++b)
    for (int n = 0; n < 16; ++n) {
      double a = -2.0 * AOM_C_PI * (double)(b * n) / (double)N;
      twr[b * 16 + n] = (float)cos(a);
      twi[b * 16 + n] = (float)sin(a);
    }
  std::vector<float> x1r(16 * W), x1i(16 * W);
  for (int y = 0; y < 16; ++y)
    for (int b = 0; b < R; ++b) {
      float outr[8], outi[8];
      aom_fft16_pruned(inr + 16 * y, ini + 16 * y, &twr[b * 16], &twi[b * 16], outr, outi);
      for (int q = 0; q < 4; ++q) {
        x1r[y * W + H + R * q + b] = outr[q];     x1i[y * W + H + R * q + b] = outi[q];
        x1r[y * W + R * q + b] = outr[4 + q];     x1i[y * W + R * q + b] = outi[4 + q];
      }
    }
  for (int c = 0; c < W; ++c)
    for (int b = 0; b < R; ++b) {
      float vr[16], vi[16], outr[8], outi[8];
      for (int n = 0; n < 16; ++n) { vr[n] = x1r[n * W + c]; vi[n] = x1i[n * W + c]; }
      aom_fft16_pruned(vr, vi, &twr[b * 16], &twi[b * 16], outr, outi);
      for (int q = 0; q < 4; ++q) {
        inten[(H + R * q + b) * W + c] = outr[q] * outr[q] + outi[q] * outi[q];
        inten[(R * q + b) * W + c] = outr[4 + q] * outr[4 + q] + outi[4 + q] * outi[4 + q];
      }
    }
}

// pre-split TF32 planes of the actor weights in the tile order of gemm_tc_kernel (gemm_tc_host.h)
long long h_pretile_floats(int n_cols_ld, int K) { return (long long)gtc_pretile_floats(n_cols_ld, K); }
void h_pretile(const float* W, int batch, long long sB, int ldb, int rows, int n_cols_ld, int K, float* out) {
  gtc_pretile_host(W, batch, sB, ldb, rows, n_cols_ld, K, out);
}

// Lattice analysis of the staged sensor kernels (wfs_lattice_host.h).  Returns null and fills geom = {cx, cy, joffx, joffy,
// c0x, c0y, GW, dm}, the padded actuator map amap_pad [GW * GW], each subaperture's window origin win [nvalid] and the
// stamp factors fac [2][WFL_NG][16]; or returns the refusal.
const char* h_wfs_lattice(const aom_config* c, const float* pup, const int* sx, const int* sy, const float* stamp,
                          const int* amap, int* geom, short* amap_pad, int* win, float* fac) {
  WfsLattice L;
  const char* why = wfl_analyse(*c, pup, sx, sy, stamp, amap, L);
  if (why) return why;
  const int g[8] = {L.cx, L.cy, L.joffx, L.joffy, L.c0x, L.c0y, L.GW, L.dm ? 1 : 0};
  for (int i = 0; i < 8; ++i) geom[i] = g[i];
  wfl_amap(*c, L, amap, amap_pad);
  for (int k = 0; k < c->nvalid; ++k) win[k] = wfl_window(*c, L, sx[k], sy[k]);
  for (int ax = 0; ax < 2; ++ax)
    for (int j = 0; j < WFL_NG; ++j)
      for (int x = 0; x < 16; ++x) fac[(ax * WFL_NG + j) * 16 + x] = wfl_factor(*c, L, stamp, ax, j, x);
  return nullptr;
}

// Digit code of the integer contraction (extrude_i8_digits.h).  Tile geometry: {OZ_SLICES, OZ_SLICES_B, OZ_LEVELS,
// OZ_LEVELS_PRODUCT, OZ_BM, OZ_BN, OZ_BK, OZ_A_TILE, OZ_B_TILE, OZ_EV_NONFINITE}.
void h_oz_constants(int* c) {
  const int v[10] = {OZ_SLICES, OZ_SLICES_B, OZ_LEVELS, OZ_LEVELS_PRODUCT, OZ_BM, OZ_BN, OZ_BK, OZ_A_TILE, OZ_B_TILE, OZ_EV_NONFINITE};
  for (int i = 0; i < 10; ++i) c[i] = v[i];
}
int h_oz_tile_offset(int r, int kk) { return (int)oz_tile_offset(r, kk); }
void h_oz_exponent(int n, const double* amax, int* e) {
  for (int i = 0; i < n; ++i) e[i] = oz_exponent(amax[i]);
}
// q [OZ_SLICES][n]: digits of x[i] * scale[i] in float32 (oz_digits_f32) and in float64 (oz_digits)
void h_oz_digits_f32(int n, const float* x, const float* scale, int* q) {
  for (int i = 0; i < n; ++i) {
    int d[OZ_SLICES];
    oz_digits_f32<OZ_SLICES>(x[i], scale[i], d);
    for (int s = 0; s < OZ_SLICES; ++s) q[(size_t)s * n + i] = d[s];
  }
}
void h_oz_digits(int n, const double* x, const double* scale, int* q) {
  for (int i = 0; i < n; ++i) {
    int d[OZ_SLICES_B];
    oz_digits<OZ_SLICES_B>(x[i], scale[i], d);
    for (int s = 0; s < OZ_SLICES_B; ++s) q[(size_t)s * n + i] = d[s];
  }
}
int h_oz_operator_finite(const float* AB, int rows, int ld, int K) { return oz_operator_finite(AB, rows, ld, K); }
void h_oz_slice_operator(const float* AB, int rows, int ld, int K, int KB, int NT, uint8_t* planes, int* ea) {
  oz_slice_operator(AB, rows, ld, K, KB, NT, planes, ea);
}
}
