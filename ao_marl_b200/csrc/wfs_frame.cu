// Host side of the Shack-Hartmann frame: which kernel serves a frame (wfs_route), the derived tables of the staged
// kernels -- wfs_frame_tma_kernel (wfs_tma.cuh) and the tcgen05 pair (wfs_umma.cuh, wfs_umma_ws.cuh) -- with their
// eligibility and TMA descriptors, and the launch of every kernel family.  Both staged generations read the mirror
// through the same lattice analysis (wfs_lattice_host.h) and lay out its tables their own way.
#include <cuda_fp16.h>
#include <math.h>
#include <new>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "dispatch.h"
#include "wfs_frame_host.h"
#include "wfs_kernels.cuh"
#include "wfs_mma.cuh"
#include "wfs_tma.cuh"
#include "wfs_umma_host.h"

struct WfsFrame {
  aom_config cfg;
  float* screen[AOM_MAX_LAYERS];
  int* err;                  // device error word of the bounded waits
  int num_sms;
  // host copies of the tables the staged kernels derive their own from; why says why the last refused preparation refused
  void* htab[AOM_T_COUNT];
  char why[160];
  // TMA-staged kernel (wfs_tma.cuh): derived tables
  int fast_state;            // 0 = not prepared, 1 = eligible, -1 = not eligible
  WfsFast fast;
  void* fast_dev[6];
  CUtensorMap fast_maps[WFT_MAX_LAYERS];
  // tcgen05 kernels (wfs_umma.cuh, wfs_umma_ws.cuh): derived tables
  int umma_state;            // 0 = not prepared, 1 = eligible, -1 = not eligible
  WfsUmmaHost umma;
  void* umma_dev[6];
};

WfsFrame* wfs_frame_create(const aom_config& c, float* const* screens, int* err, int num_sms) {
  WfsFrame* s = new (std::nothrow) WfsFrame();
  if (!s) return nullptr;
  s->cfg = c;
  for (int l = 0; l < AOM_MAX_LAYERS; ++l) s->screen[l] = screens[l];
  s->err = err;
  s->num_sms = num_sms;
  return s;
}

void wfs_frame_destroy(WfsFrame* s) {
  if (!s) return;
  for (void* b : s->fast_dev) cudaFree(b);
  for (void* b : s->umma_dev) cudaFree(b);
  for (void* h : s->htab) free(h);
  delete s;
}

bool wfs_frame_set_table(WfsFrame* s, int table, const void* host, size_t nbytes) {
  if (table != AOM_T_MPUPIL && table != AOM_T_SUB_X0 && table != AOM_T_SUB_Y0 && table != AOM_T_STAMP1D &&
      table != AOM_T_ACT_MAP && table != AOM_T_HALFXY && table != AOM_T_TT_PLANES)
    return true;
  free(s->htab[table]);
  s->htab[table] = malloc(nbytes ? nbytes : 4);
  if (!s->htab[table]) return false;
  memcpy(s->htab[table], host, nbytes);
  s->fast_state = 0;     // derived tables of the staged sensor kernels are rebuilt on the next frame
  s->umma_state = 0;
  return true;
}

// ---- staged kernels: eligibility, derived tables, TMA descriptors ----
static void split_pair(double a, double b, int lo_part, uint32_t& out) {
  const float ah = __half2float(__float2half_rn((float)a)), bh = __half2float(__float2half_rn((float)b));
  const __half2 h = lo_part ? __floats2half2_rn((float)(a - (double)ah), (float)(b - (double)bh)) : __floats2half2_rn(ah, bh);
  memcpy(&out, &h, 4);
}

// W[n][i] = exp(-2 pi i n F(i) / 64), F = the 32 kept frequencies (0..15, 48..63); part 0 = real, 1 = imaginary
static double wft_w(int n, int i, int part) {
  const int F = (i < 16) ? i : i + 32;
  const int ang = (n * F) & 63;
  const double th = -2.0 * M_PI * (double)ang / 64.0;
  return part ? sin(th) : cos(th);
}

typedef CUresult (*aom_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// A staged kernel cannot serve this configuration: its state becomes -1 and why says why.  Returns cudaSuccess.
static cudaError_t staged_refuse(WfsFrame* s, int& state, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(s->why, sizeof(s->why), fmt, ap);
  va_end(ap);
  state = -1;
  return cudaSuccess;
}

// The lattice analysis of the uploaded host tables: null, or why the staged kernels cannot serve them
static const char* staged_lattice(WfsFrame* s, WfsLattice& L) {
  return wfl_analyse(s->cfg, (const float*)s->htab[AOM_T_MPUPIL], (const int*)s->htab[AOM_T_SUB_X0],
                     (const int*)s->htab[AOM_T_SUB_Y0], (const float*)s->htab[AOM_T_STAMP1D],
                     (const int*)s->htab[AOM_T_ACT_MAP], L);
}

// One 3-D map [E][N][N] per screen layer, box bw x bh x 1, zero fill outside.  False: refused (state, why).
static bool encode_screen_maps(WfsFrame* s, CUtensorMap* maps, cuuint32_t bw, cuuint32_t bh, int& state) {
  const aom_config& c = s->cfg;
  if (c.n_layers == 0) return true;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    staged_refuse(s, state, "cuTensorMapEncodeTiled not available");
    return false;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    const cuuint64_t N = (cuuint64_t)c.screen_dim[l];
    const cuuint64_t dims[3] = {N, N, (cuuint64_t)c.n_env};
    const cuuint64_t strides[2] = {N * 4, N * N * 4};
    const cuuint32_t box[3] = {bw, bh, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = ((aom_encode_tiled_fn)fn)(&maps[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, s->screen[l], dims, strides, box,
                                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      staged_refuse(s, state, "cuTensorMapEncodeTiled failed (%d)", (int)r);
      return false;
    }
  }
  return true;
}

// Copies the six host tables src[i] of bytes[i] into new device buffers dev[i]
static cudaError_t upload_tables(void* (&dev)[6], const void* const (&src)[6], const size_t (&bytes)[6]) {
  cudaError_t ce = cudaSuccess;
  for (int i = 0; i < 6 && ce == cudaSuccess; ++i) {
    ce = cudaMalloc(&dev[i], bytes[i]);
    if (ce == cudaSuccess) ce = cudaMemcpy(dev[i], src[i], bytes[i], cudaMemcpyHostToDevice);
  }
  return ce;
}

static cudaError_t wfs_fast_prepare(WfsFrame* s) {
  const aom_config& c = s->cfg;
  if (s->fast_state != 0) return cudaSuccess;
  for (void*& b : s->fast_dev) { cudaFree(b); b = nullptr; }
  WfsLattice L;
  if (const char* why = staged_lattice(s, L)) return staged_refuse(s, s->fast_state, "%s", why);
  const float* pup = (const float*)s->htab[AOM_T_MPUPIL];
  const int* sx = (const int*)s->htab[AOM_T_SUB_X0];
  const int* sy = (const int*)s->htab[AOM_T_SUB_Y0];
  const float* stamp = (const float*)s->htab[AOM_T_STAMP1D];
  const int nv = c.nvalid, GW = L.GW;
  uint2* h_sub = (uint2*)malloc((size_t)nv * sizeof(uint2));
  unsigned char* h_pm = (unsigned char*)malloc((size_t)nv * 32);
  short* h_amap = (short*)malloc((size_t)GW * GW * sizeof(short));
  float h_fxy[2 * WFT_NG * 16];
  uint4 h_c1[8 * 32], h_c2[12 * 32];
  const bool ok = h_sub && h_pm && h_amap;
  if (ok) {
    wfl_amap(c, L, (const int*)s->htab[AOM_T_ACT_MAP], h_amap);
    for (int k = 0; k < nv; ++k) {
      h_sub[k] = make_uint2(((uint32_t)sy[k] << 16) | (uint32_t)sx[k], (uint32_t)wfl_window(c, L, sx[k], sy[k]));
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, q = lane & 3;
        unsigned m = 0;
        for (int r = 0; r < 2; ++r)
          for (int cc = 0; cc < 4; ++cc)
            if (pup[(size_t)(sy[k] + 2 * g + r) * c.n + sx[k] + 4 * q + cc] != 0.f) m |= 1u << (r * 4 + cc);
        h_pm[(size_t)k * 32 + lane] = (unsigned char)m;
      }
    }
    for (int ax = 0; ax < 2; ++ax)
      for (int j = 0; j < WFT_NG; ++j)
        for (int x = 0; x < 16; ++x) h_fxy[(ax * WFT_NG + j) * 16 + x] = wfl_factor(c, L, stamp, ax, j, x);
    // stage-1 A fragments: row r of m-tile mt <-> kept frequency 16 mt + 2 (r & 7) + (r >> 3); k <-> x = sigma(k)
    auto sigma = [](int kk) { return kk < 8 ? 4 * (kk >> 1) + (kk & 1) : 4 * ((kk - 8) >> 1) + 2 + (kk & 1); };
    auto yk = [](int kk) { return kk < 8 ? 2 * kk : 2 * (kk - 8) + 1; };
    for (int mt = 0; mt < 2; ++mt)
      for (int part = 0; part < 2; ++part)
        for (int hl = 0; hl < 2; ++hl)
          for (int lane = 0; lane < 32; ++lane) {
            const int g = lane >> 2, q = lane & 3;
            const int rows[2] = {g, g + 8};
            const int ks[4] = {2 * q, 2 * q + 1, 2 * q + 8, 2 * q + 9};
            uint32_t w[4];
            for (int reg = 0; reg < 4; ++reg) {      // a0 (g; 2q..) a1 (g+8; 2q..) a2 (g; 2q+8..) a3 (g+8; 2q+8..)
              const int r = rows[reg & 1], fi = 16 * mt + 2 * (r & 7) + (r >> 3);
              const int k0 = ks[(reg >> 1) * 2], k1 = ks[(reg >> 1) * 2 + 1];
              split_pair(wft_w(sigma(k0), fi, part), wft_w(sigma(k1), fi, part), hl, w[reg]);
            }
            h_c1[((mt * 2 + part) * 2 + hl) * 32 + lane] = make_uint4(w[0], w[1], w[2], w[3]);
          }
    // stage-2 B fragments: k <-> y = yk(k), n = g <-> kept frequency 8 b + g
    for (int b = 0; b < 4; ++b)
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, q = lane & 3;
        const int ks[4] = {2 * q, 2 * q + 1, 2 * q + 8, 2 * q + 9};
        uint32_t hi[4], lo[4], nh[2], nl[2];
        for (int reg = 0; reg < 4; ++reg) {        // {Wr b0, Wr b1, Wi b0, Wi b1}
          const int part = reg >> 1, k0 = ks[(reg & 1) * 2], k1 = ks[(reg & 1) * 2 + 1];
          split_pair(wft_w(yk(k0), 8 * b + g, part), wft_w(yk(k1), 8 * b + g, part), 0, hi[reg]);
          split_pair(wft_w(yk(k0), 8 * b + g, part), wft_w(yk(k1), 8 * b + g, part), 1, lo[reg]);
        }
        for (int h = 0; h < 2; ++h) { nh[h] = hi[2 + h] ^ 0x80008000u; nl[h] = lo[2 + h] ^ 0x80008000u; }
        h_c2[(b * 3 + 0) * 32 + lane] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        h_c2[(b * 3 + 1) * 32 + lane] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        h_c2[(b * 3 + 2) * 32 + lane] = make_uint4(nh[0], nh[1], nl[0], nl[1]);
      }
  }
  const void* const srcs[6] = {h_sub, h_amap, h_pm, h_c1, h_c2, h_fxy};
  const size_t sizes[6] = {(size_t)nv * sizeof(uint2), (size_t)GW * GW * sizeof(short), (size_t)nv * 32,
                           sizeof(h_c1), sizeof(h_c2), sizeof(h_fxy)};
  const cudaError_t ce = ok ? upload_tables(s->fast_dev, srcs, sizes) : cudaSuccess;
  free(h_sub); free(h_pm); free(h_amap);
  if (ce != cudaSuccess) return ce;
  if (!ok) return staged_refuse(s, s->fast_state, "out of host memory");
  if (!encode_screen_maps(s, s->fast_maps, WFT_TILE_W, WFT_TILE_H, s->fast_state)) return cudaSuccess;
  WfsFast& f = s->fast;
  f.sub = (const uint2*)s->fast_dev[0];
  f.amap = (const short*)s->fast_dev[1];
  f.pmask = (const unsigned char*)s->fast_dev[2];
  f.c1 = (const uint4*)s->fast_dev[3];
  f.c2 = (const uint4*)s->fast_dev[4];
  f.fxy = (const float*)s->fast_dev[5];
  f.GW = GW;
  f.sub_in_smem = (nv <= 1280) ? 1 : 0;
  f.err = s->err;
  s->fast_state = 1;
  return cudaSuccess;
}

static void umma_put_half(unsigned short* tile_hi, unsigned short* tile_lo, int n, int kk, double v) {
  // UMMA canonical K-major no-swizzle layout: 8-row x 16-byte core matrices, LBO 128 B, SBO 512 B (K = 32 halves)
  const __half hi = __float2half_rn((float)v);
  const __half lo = __float2half_rn((float)(v - (double)__half2float(hi)));
  const size_t off = (size_t)(n >> 3) * 512 + (size_t)(kk >> 3) * 128 + (size_t)(n & 7) * 16 + (size_t)(kk & 7) * 2;
  memcpy((unsigned char*)tile_hi + off, &hi, 2);
  memcpy((unsigned char*)tile_lo + off, &lo, 2);
}

// The tcgen05 kernels also need a full group of subapertures and the analytic half-pixel phasor; their tables are in the
// (h, y) lane layout, with the operand tiles of the two DFT stages and 20 x 17 TMA boxes.
static cudaError_t wfs_umma_prepare(WfsFrame* s) {
  const aom_config& c = s->cfg;
  if (s->umma_state != 0) return cudaSuccess;
  for (void*& b : s->umma_dev) { cudaFree(b); b = nullptr; }
  WfsLattice L;
  if (const char* why = staged_lattice(s, L)) return staged_refuse(s, s->umma_state, "%s", why);
  if (c.nvalid < WU_WARPS) return staged_refuse(s, s->umma_state, "fewer than %d subapertures", WU_WARPS);
  const float* hxy = (const float*)s->htab[AOM_T_HALFXY];
  if (!hxy) return staged_refuse(s, s->umma_state, "half-pixel phasor table not uploaded");
  for (int i = 0; i < 16; ++i)
    for (int j = 0; j < 16; ++j)
      if (fabs((double)hxy[i * 16 + j] - M_PI * (double)(i + j) / 64.0) > 2e-6)
        return staged_refuse(s, s->umma_state, "half-pixel phasor is not pi (x + y) / Nfft");
  const float* pup = (const float*)s->htab[AOM_T_MPUPIL];
  const int* sx = (const int*)s->htab[AOM_T_SUB_X0];
  const int* sy = (const int*)s->htab[AOM_T_SUB_Y0];
  const float* stamp = (const float*)s->htab[AOM_T_STAMP1D];
  const int nv = c.nvalid, GW = L.GW;
  uint2* h_sub = (uint2*)malloc((size_t)nv * sizeof(uint2));
  uint32_t* h_pm = (uint32_t*)malloc((size_t)nv * 32 * sizeof(uint32_t));
  short* h_amap = (short*)malloc((size_t)GW * GW * sizeof(short));
  unsigned short h_b1[WU_B_BYTES] = {}, h_b2[WU_B_BYTES] = {};     // [hi, lo] tiles of WU_B_BYTES bytes each
  float h_fxy[2 * WU_NG * 16];
  const bool ok = h_sub && h_pm && h_amap;
  if (ok) {
    wfl_amap(c, L, (const int*)s->htab[AOM_T_ACT_MAP], h_amap);
    for (int k = 0; k < nv; ++k) {
      bool full = true;
      for (int lane = 0; lane < 32; ++lane) {
        const int yy = lane & 15, hh = lane >> 4;
        unsigned m = 0;
        for (int cc = 0; cc < 8; ++cc)
          if (pup[(size_t)(sy[k] + yy) * c.n + sx[k] + 8 * hh + cc] != 0.f) m |= 1u << cc;
        h_pm[(size_t)k * 32 + lane] = m;
        full = full && m == 0xffu;
      }
      h_sub[k] = make_uint2(((uint32_t)sy[k] << 16) | (uint32_t)sx[k],
                            (uint32_t)wfl_window(c, L, sx[k], sy[k]) | (full ? 0x80000000u : 0u));
    }
    // x stamp factors [j][x], y stamp factors transposed [y][j]
    for (int j = 0; j < WU_NG; ++j)
      for (int x = 0; x < 16; ++x) {
        h_fxy[j * 16 + x] = wfl_factor(c, L, stamp, 0, j, x);
        h_fxy[WU_NG * 16 + x * WU_NG + j] = wfl_factor(c, L, stamp, 1, j, x);
      }
    // stage 1: B1[n = 32 ro + fx][k = 16 ri + x]:  Tr = Wr Xr - Wi Xi ; Ti = Wi Xr + Wr Xi
    // stage 2: B2[n = 2 fy + po][k = 16 ro + y]:   Yr = Tr Wr - Ti Wi ; Yi = Tr Wi + Ti Wr
    unsigned short* b1_lo = (unsigned short*)((unsigned char*)h_b1 + WU_B_BYTES);
    unsigned short* b2_lo = (unsigned short*)((unsigned char*)h_b2 + WU_B_BYTES);
    for (int n = 0; n < 64; ++n)
      for (int kk = 0; kk < 32; ++kk) {
        {
          const int ro = n >> 5, fx = n & 31, ri = kk >> 4, x = kk & 15;
          const double wr = wft_w(x, fx, 0), wi = wft_w(x, fx, 1);
          umma_put_half(h_b1, b1_lo, n, kk, ro == 0 ? (ri == 0 ? wr : -wi) : (ri == 0 ? wi : wr));
        }
        {
          const int fy = n >> 1, po = n & 1, ro = kk >> 4, yy = kk & 15;
          const double wr = wft_w(yy, fy, 0), wi = wft_w(yy, fy, 1);
          umma_put_half(h_b2, b2_lo, n, kk, po == 0 ? (ro == 0 ? wr : -wi) : (ro == 0 ? wi : wr));
        }
      }
  }
  const void* const srcs[6] = {h_sub, h_amap, h_pm, h_b1, h_b2, h_fxy};
  const size_t sizes[6] = {(size_t)nv * sizeof(uint2), (size_t)GW * GW * sizeof(short), (size_t)nv * 32 * sizeof(uint32_t),
                           sizeof(h_b1), sizeof(h_b2), sizeof(h_fxy)};
  const cudaError_t ce = ok ? upload_tables(s->umma_dev, srcs, sizes) : cudaSuccess;
  free(h_sub); free(h_pm); free(h_amap);
  if (ce != cudaSuccess) return ce;
  if (!ok) return staged_refuse(s, s->umma_state, "out of host memory");
  if (!encode_screen_maps(s, s->umma.maps, WU_TILE_W, WU_TILE_H, s->umma_state)) return cudaSuccess;
  WfsUmmaTables& f = s->umma.f;
  memset(&f, 0, sizeof(f));
  f.sub = (const uint2*)s->umma_dev[0];
  f.amap = (const short*)s->umma_dev[1];
  f.pmask = (const uint32_t*)s->umma_dev[2];
  f.b1 = (const uint4*)s->umma_dev[3];
  f.b2 = (const uint4*)s->umma_dev[4];
  f.fxy = (const float*)s->umma_dev[5];
  f.GW = GW;
  f.err = s->err;
  s->umma_state = 1;
  return cudaSuccess;
}

template <int FULL, int NL>
static cudaError_t wfs_fast_launch_t(WfsFrame* s, const WfsParams& p, cudaStream_t st) {
  const long long total = (long long)p.E * p.nvalid;
  // contiguous ranges of work items per CTA: about 8 waves of resident CTAs per SM, at least 16 items per warp
  long long grid = (long long)s->num_sms * WFT_MIN_CTAS * 8;
  long long ipc = (total + grid - 1) / grid;
  if (ipc < 16 * WFT_WARPS) ipc = 16 * WFT_WARPS;
  ipc = (ipc + WFT_WARPS - 1) / WFT_WARPS * WFT_WARPS;
  grid = (total + ipc - 1) / ipc;
  WfsTmaParams P;
  memset(&P, 0, sizeof(P));
  P.p = p;
  P.f = s->fast;
  P.f.items_per_cta = ipc;
  for (int l = 0; l < NL; ++l) P.maps[l] = s->fast_maps[l];
  const size_t smem = wft_smem_bytes<NL>(P.f.GW, P.f.sub_in_smem ? p.nvalid : 0);
  cudaError_t e = cudaFuncSetAttribute(wfs_frame_tma_kernel<FULL, NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) wfs_frame_tma_kernel<FULL, NL><<<(unsigned)grid, WFT_WARPS * 32, smem, st>>>(P);
  return e;
}

// The sensor kernel that serves a frame: its family with its compile-time choices, and whether the frame is refused
enum WfsFamily { WFS_WS, WFS_UMMA, WFS_TMA, WFS_MMA, WFS_SIMT };
static const char* const wfs_kernel_names[] = {"wfs_frame_ws_kernel", "wfs_frame_umma_kernel", "wfs_frame_tma_kernel",
                                               "wfs_frame_mma_kernel", "wfs_frame_kernel"};
struct WfsRoute {
  WfsFamily family;
  bool full, pe, ne;     // fp32-grade products in both DFT stages; per-environment winds; per-environment sensor values
  int nl, r;             // layers of the instantiation (mma: 0, 1 or 3, else -1: its generic form); simt: Nfft / 16
  const char* refused;   // not null: the frame is refused with this message (family still names the path's kernel)
};

static int report(char (&err)[512], int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err, sizeof(err), fmt, ap);
  va_end(ap);
  return code;
}

// Routes a frame of parameters p (fill_wfs_params) on path, noisy when any environment draws noise in it, with its image
// kept when p.bincube is set.  Prepares the tables of a staged kernel on first use, and the round-1 kernel's only when
// the route can reach it.
static int wfs_route(WfsFrame* s, const WfsParams& p, int path, bool noisy, WfsRoute& r, char (&err)[512]) {
  const aom_config& c = s->cfg;
  const bool umma = (path == AOM_WFS_UMMA || path == AOM_WFS_UMMA_FAST || path == AOM_WFS_UMMA_WS);
  const bool staged = umma || path == AOM_WFS_MMA_STAGED || path == AOM_WFS_MMA_STAGED_FAST;
  memset(&r, 0, sizeof(r));
  r.full = !(path == AOM_WFS_UMMA_FAST || path == AOM_WFS_MMA_STAGED_FAST);
  r.nl = p.n_layers;
  r.pe = p.wind != nullptr;
  r.ne = p.noise_env || p.nph_env;
  if (c.nfft != 64 || path == AOM_WFS_SIMT) {
    r.family = WFS_SIMT;
    r.r = c.nfft / 16;
    return AOM_OK;
  }
  if (umma) {
    cudaError_t e = wfs_umma_prepare(s);
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "wfs_umma_prepare: %s", cudaGetErrorString(e));
  }
  if (umma && s->umma_state == 1) {
    // the specialised-warp kernel serves every frame without noise and kept image (it reads neither noise nor photon
    // count); the others go to the fused kernel, in its per-environment form when per-environment values are in force
    r.family = (path == AOM_WFS_UMMA_WS && !noisy && !p.bincube) ? WFS_WS : WFS_UMMA;
    if (r.family == WFS_WS) r.ne = false;
    return AOM_OK;
  }
  if (staged) {
    cudaError_t e = wfs_fast_prepare(s);
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "wfs_fast_prepare: %s", cudaGetErrorString(e));
  }
  r.family = (staged && s->fast_state == 1) ? WFS_TMA : WFS_MMA;
  if (r.family == WFS_MMA && r.nl != 0 && r.nl != 1 && r.nl != 3) r.nl = -1;
  // the round-1 kernels have no per-environment form
  r.refused = p.frame0 ? "staggered environments (aom_reset_envs) are not implemented in the round-1 sensor kernels "
                         "(wfs_frame_tma_kernel, wfs_frame_mma_kernel) until the next aom_reset: use the umma, umma_ws or simt path"
            : p.wind ? "per-environment wind is not implemented in the round-1 sensor kernels (wfs_frame_tma_kernel, "
                       "wfs_frame_mma_kernel): use the umma, umma_ws or simt path"
            : r.ne ? "per-environment sensor noise and photon counts are not implemented in the round-1 sensor kernels "
                     "(wfs_frame_tma_kernel, wfs_frame_mma_kernel): use the umma, umma_ws or simt path"
            : nullptr;
  return AOM_OK;
}

int wfs_frame_launch(WfsFrame* s, const WfsParams& p, int path, bool noisy, cudaEvent_t start, cudaStream_t st,
                     char (&err)[512]) {
  WfsRoute r;
  int rc = wfs_route(s, p, path, noisy, r, err);
  if (rc) return rc;
  if (r.refused) return report(err, AOM_ERR_UNSUPPORTED, "%s", r.refused);
  if (start) {
    cudaError_t e = cudaEventRecord(start, st);
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "cudaEventRecord failed: %s", cudaGetErrorString(e));
  }
  const long long total = (long long)p.E * p.nvalid;
  const long long blocks = (total + WFS_WARPS - 1) / WFS_WARPS;
  const long long cap = (long long)s->num_sms * 2 * 8;      // 2 resident CTAs per SM, 8 waves of work each
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (r.family == WFS_WS || r.family == WFS_UMMA) {
    WfsParams q = p;
    if (r.family == WFS_WS) { q.noise = -1.f; q.noise_env = nullptr; q.nph_env = nullptr; }
    cudaError_t e = wfs_umma_launch(q, s->umma, s->num_sms, r.family == WFS_WS, r.full, r.ne, st);
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "wfs_umma_launch: %s", cudaGetErrorString(e));
  } else if (r.family == WFS_TMA) {
    cudaError_t e = cudaSuccess;
    const bool served = with<0, 1, 2, 3, 4>(p.n_layers, [&](auto NL) {
      with<false, true>(r.full, [&](auto FULL) { e = wfs_fast_launch_t<FULL, NL>(s, p, st); });
    });
    if (!served) return report(err, AOM_ERR_UNSUPPORTED, "wfs_fast_launch: %d layers", p.n_layers);
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "cudaFuncSetAttribute(wfs_frame_tma_kernel): %s", cudaGetErrorString(e));
  } else if (r.family == WFS_MMA) {
    with<0, 1, 3, -1>(r.nl, [&](auto NL) {
      with<false, true>(r.full, [&](auto FULL) { wfs_frame_mma_kernel<FULL, NL><<<grid, WFM_WARPS * 32, 0, st>>>(p); });
    });
  } else {
    // SIMT frame: Nfft / 16, per-environment winds, per-environment sensor values
    cudaError_t e = cudaSuccess;
    with<4, 8>(r.r, [&](auto R) {
      with<false, true>(r.pe, [&](auto PE) {
        with<false, true>(r.ne, [&](auto NE) {
          const size_t smem = wfs_smem_bytes<R>();
          e = cudaFuncSetAttribute(wfs_frame_kernel<R, PE, NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
          if (e == cudaSuccess) wfs_frame_kernel<R, PE, NE><<<grid, WFS_WARPS * 32, smem, st>>>(p);
        });
      });
    });
    if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "cudaFuncSetAttribute(wfs_frame_kernel): %s", cudaGetErrorString(e));
  }
  return AOM_OK;
}

const char* wfs_frame_kernel_name(WfsFrame* s, int path, char (&err)[512]) {
  // the route of a noise-free frame without kept image; the per-environment state does not change its family, so the
  // fields the route reads for it stay empty (and a refusal it would cause is not reported)
  const WfsParams p{};
  WfsRoute r;
  if (wfs_route(s, p, path, false, r, err) != AOM_OK) return "";
  if (r.family == WFS_MMA && path != AOM_WFS_MMA_REG) snprintf(err, sizeof(err), "staged sensor kernels not eligible: %s", s->why);
  return wfs_kernel_names[r.family];
}
