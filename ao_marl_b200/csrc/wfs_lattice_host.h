// Host side of the actuator lattice the staged sensor kernels (wfs_tma.cuh, wfs_umma.cuh, wfs_umma_ws.cuh) read the mirror
// through: plain C++, no CUDA, so that the CPU test harness (tests/cpu_kernels/harness.cpp) checks the same code the library
// runs when it prepares those kernels.
//
// With a 16-pixel actuator pitch and every subaperture at the same offset from the lattice, the mirror surface over a
// 16 x 16 subaperture is the separable sum over a WFL_NG x WFL_NG window of lattice cells:
//   dm(x, y) = sum_{jx, jy} volts[amap[window + jy * GW + jx]] * fx(jx, x) * fy(jy, y)
// where amap is the actuator map padded by WFL_PAD cells on every side and the stamp factors fx, fy are the same for every
// subaperture.
#pragma once
#include "../../include/aomarl.h"

#define WFL_NG 4                           // lattice cells per axis whose stamp meets one subaperture
#define WFL_PAD 4                          // border of the padded actuator map
#define WFL_MAX_LAYERS 4                   // screen layers the staged kernels sample
#define WFL_STR_(x) #x
#define WFL_STR(x) WFL_STR_(x)

struct WfsLattice {
  int cx, cy;          // subaperture origin in the mirror support, relative to the lattice, modulo the pitch
  int joffx, joffy;    // window cell 0 is lattice cell m - joff, m = (X0 - cx) / 16
  int c0x, c0y;        // stamp index of pixel 0 in window cell 0
  int GW;              // side of the padded actuator map
  bool dm;             // stamp and actuator map uploaded
};

// Window origin (column gxl, row gyl of the padded map) of the subaperture at (sx, sy) in the pupil frame
static inline void wfl_origin(const aom_config& c, const WfsLattice& L, int sx, int sy, int& gxl, int& gyl) {
  gxl = (sx + c.pzt_off - c.pzt_i1_0 - L.cx) / 16 - L.joffx + WFL_PAD;   // exact multiples of 16
  gyl = (sy + c.pzt_off - c.pzt_j1_0 - L.cy) / 16 - L.joffy + WFL_PAD;
}

// Its index in the padded map (0 without mirror tables)
static inline int wfl_window(const aom_config& c, const WfsLattice& L, int sx, int sy) {
  int gxl = 0, gyl = 0;
  if (L.dm) wfl_origin(c, L, sx, sy, gxl, gyl);
  return gyl * L.GW + gxl;
}

// Stamp factor of window cell j at pixel x of the subaperture, along x (axis 0) or y (axis 1)
static inline float wfl_factor(const aom_config& c, const WfsLattice& L, const float* stamp, int axis, int j, int x) {
  const int a = (axis ? L.c0y : L.c0x) + x - 16 * j;
  return (L.dm && a >= 0 && a < c.stamp_size) ? stamp[a] : 0.f;
}

// The padded actuator map [GW * GW]: actuator index or -1
static inline void wfl_amap(const aom_config& c, const WfsLattice& L, const int* amap, short* out) {
  for (int i = 0; i < L.GW * L.GW; ++i) out[i] = -1;
  if (L.dm)
    for (int gy = 0; gy < c.pzt_grid_n; ++gy)
      for (int gx = 0; gx < c.pzt_grid_n; ++gx) out[(gy + WFL_PAD) * L.GW + gx + WFL_PAD] = (short)amap[gy * c.pzt_grid_n + gx];
}

// Whether the staged kernels can serve configuration c with the host tables pup (MPUPIL), sx / sy (SUB_X0 / SUB_Y0), stamp
// (STAMP1D) and amap (ACT_MAP; stamp and amap may both be null: no mirror term).  Fills L and returns null, or returns why not.
static inline const char* wfl_analyse(const aom_config& c, const float* pup, const int* sx, const int* sy, const float* stamp,
                                      const int* amap, WfsLattice& L) {
  L = WfsLattice{};
  if (c.nfft != 64 || c.nrebin != 2) return "Nfft != 64";
  if (c.n_layers > WFL_MAX_LAYERS) return "more than " WFL_STR(WFL_MAX_LAYERS) " layers";
  if (c.pzt_pitch != 16) return "actuator pitch is not 16 pixels";
  if (c.nvalid > 65535 / 256 * 256 || c.n > 65535) return "geometry too large for the packed tables";
  if ((c.tt_dim & 3) || c.tt_dim <= 0) return "tip-tilt support not a multiple of 4";
  if (!pup || !sx || !sy) return "sensor tables not uploaded";
  L.dm = stamp && amap;
  for (int l = 0; l < c.n_layers; ++l)
    if (c.screen_dim[l] & 3) return "screen side not a multiple of 4";
  for (size_t i = 0; i < (size_t)c.n * c.n; ++i)
    if (pup[i] != 0.f && pup[i] != 1.f) return "pupil transmission is not binary";
  for (int k = 0; k < c.nvalid; ++k) {
    if (sx[k] < 0 || sy[k] < 0 || sx[k] + 16 > c.n || sy[k] + 16 > c.n) return "subaperture outside the pupil frame";
    if ((sx[k] + c.tt_off) & 3) return "tip-tilt rows not 16-byte aligned";
    const int mx = (((sx[k] + c.pzt_off - c.pzt_i1_0) % 16) + 16) % 16, my = (((sy[k] + c.pzt_off - c.pzt_j1_0) % 16) + 16) % 16;
    if (k == 0) { L.cx = mx; L.cy = my; }
    if (mx != L.cx || my != L.cy) return "subapertures not aligned with the actuator lattice";
  }
  // window cells j = 0 .. NG-1 from gx_lo = m - joff; stamp index a = c0 + x - 16 j
  auto axis = [&](int cm, int& joff, int& c0) {
    const int num = cm - (c.stamp_size - 1);             // ceil(num / 16) = -joff
    joff = -((num >= 0) ? (num + 15) / 16 : -((-num) / 16));
    c0 = cm + 16 * joff;
    return (c0 + 15) / 16 + 1;                           // cells the stamp spans
  };
  if (L.dm && (axis(L.cx, L.joffx, L.c0x) > WFL_NG || axis(L.cy, L.joffy, L.c0y) > WFL_NG))
    return "stamp spans more than " WFL_STR(WFL_NG) " lattice cells";
  L.GW = c.pzt_grid_n + 2 * WFL_PAD;
  if ((size_t)L.GW * L.GW * 2 > 16384) return "actuator lattice too large";
  if (L.dm) {
    // actuator indices fit a short, every window lies inside the padded map
    for (int i = 0; i < c.pzt_grid_n * c.pzt_grid_n; ++i)
      if (amap[i] > 32767) return "derived tables out of range";
    for (int k = 0; k < c.nvalid; ++k) {
      int gxl, gyl;
      wfl_origin(c, L, sx[k], sy[k], gxl, gyl);
      if (gxl < 0 || gyl < 0 || gxl + WFL_NG > L.GW || gyl + WFL_NG > L.GW) return "derived tables out of range";
    }
  }
  return nullptr;
}
