// Host side of the turbulence layers: the screens, the wind state and the extrusion (atmos_kernels.cuh, extrude_i8.cuh,
// and the float32 FFMA GEMM for the cross-check path).  The conditions, keys and tables stay the context's and are read
// through AtmosLinks.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "atmos_host.h"
#include "atmos_kernels.cuh"
#include "dalloc.h"
#include "dispatch.h"
#include "extrude_i8_host.h"
#include "gemm_host.h"

struct Atmos {
  aom_config cfg;
  AtmosLinks in;
  float* screen[AOM_MAX_LAYERS];
  int* ox[AOM_MAX_LAYERS];
  int* oy[AOM_MAX_LAYERS];
  uint32_t* ext_count[AOM_MAX_LAYERS];
  double accx[AOM_MAX_LAYERS], accy[AOM_MAX_LAYERS];
  // per-environment winds (aom_set_layer_wind).  While wind_pe is set every layer keeps one accumulator per environment
  // on the device (wind_state_kernel) and in a host mirror that only sizes the extrusion passes; the extrusion and
  // sampling kernels run their per-environment instantiations.  Otherwise accx / accy above hold the state.
  bool wind_pe;
  double* wind_acc;            // device [L][2][E] accumulators (x, y)
  int* wind_steps;             // device [L][2][E] whole-pixel counts of the last frame (x, y)
  WindRec* wind_rec;           // device [L][E] offsets for the samplers
  double* wind_hacc;           // host mirror of wind_acc
  int wind_passes[AOM_MAX_LAYERS][2];   // extrusion passes of the last frame: max over the batch of |count| (x, y)
  int wind_box[AOM_MAX_LAYERS][4];      // min / max over the batch of ix, then of iy (pupil footprint check)
  double* snap_acc;            // device [L][2][E] accumulators of loaded records (aom_load_envs)
  // float32 FFMA extrusion: gathered inputs, reference pixels, new lines
  float *Z, *zref, *newcol;
  int ldz_max, ldn_max;
  // exact integer extrusion (extrude_i8.cuh): digit planes of each layer's [A | B], and the scratch of the stream the
  // extrusion runs on (aom_step's second stream)
  OzOperator ab[AOM_MAX_LAYERS];
  OzScratch oz;
};

static int report(char (&err)[512], int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err, sizeof(err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t _e = (call);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return report(err, AOM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define KCHECK()                                                                                  \
  do {                                                                                            \
    ++*a->in.launches;                                                                            \
    cudaError_t _e = cudaGetLastError();                                                          \
    if (_e != cudaSuccess)                                                                        \
      return report(err, AOM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define NEED(t, i)                                                                     \
  do {                                                                                 \
    if (!a->in.tab[t][i]) return report(err, AOM_ERR_STATE, "table %s[%d] not uploaded", #t, i); \
  } while (0)

static const EnvCond& cond(const Atmos* a, int k, int l) { return a->in.cond[k][l]; }

int atmos_create(const aom_config& c, const AtmosLinks& links, Atmos** out, char (&err)[512]) {
  Atmos* a = (Atmos*)calloc(1, sizeof(Atmos));
  *out = a;
  if (!a) return report(err, AOM_ERR_INVALID, "out of host memory");
  a->cfg = c;
  a->in = links;
  const size_t E = c.n_env;
  for (int l = 0; l < c.n_layers; ++l) {
    size_t N = c.screen_dim[l];
    CU(dalloc(&a->screen[l], E * N * N));
    CU(dalloc(&a->ox[l], E));
    CU(dalloc(&a->oy[l], E));
    CU(dalloc(&a->ext_count[l], E));
    int ldz = AOM_LD(c.stencil_size[l] + (int)N);
    if (ldz > a->ldz_max) a->ldz_max = ldz;
    if (AOM_LD((int)N) > a->ldn_max) a->ldn_max = AOM_LD((int)N);
  }
  if (c.n_layers > 0) {
    CU(dalloc(&a->Z, E * a->ldz_max));
    CU(dalloc(&a->zref, E));
    CU(dalloc(&a->newcol, E * a->ldn_max));
  }
  return AOM_OK;
}

void atmos_destroy(Atmos* a) {
  if (!a) return;
  for (int l = 0; l < AOM_MAX_LAYERS; ++l) {
    cudaFree(a->screen[l]); cudaFree(a->ox[l]); cudaFree(a->oy[l]); cudaFree(a->ext_count[l]);
    oz_operator_free(a->ab[l]);
  }
  cudaFree(a->wind_acc); cudaFree(a->wind_steps); cudaFree(a->wind_rec); free(a->wind_hacc);
  cudaFree(a->snap_acc); cudaFree(a->Z); cudaFree(a->zref); cudaFree(a->newcol);
  oz_scratch_free(a->oz);
  free(a);
}

AtmosLayer atmos_layer(const Atmos* a, int l) { return AtmosLayer{a->screen[l], a->ox[l], a->oy[l], a->ext_count[l]}; }

int atmos_set_table(Atmos* a, int table, int index, const void* host, char (&err)[512]) {
  if (table != AOM_T_AB) return AOM_OK;
  const int N = a->cfg.screen_dim[index], K = a->cfg.stencil_size[index] + N;
  return oz_operator_upload(a->ab[index], (const float*)host, N, AOM_LD(K), K, err);
}

// ---------------------------------------------------------------------------------------------
// steps != null: per-environment winds -- pass `pass` of the signed counts steps [E] of this axis (`sign` unused).
// envs != null: only the K environments envs[0..K) (device), compacted into the first K rows of the scratch and the
// contraction (the start-up of aom_reset_envs).
static int extrude_once(Atmos* a, int l, int axis, int sign, cudaStream_t st, char (&err)[512], const int* steps = nullptr,
                        int pass = 0, const int* envs = nullptr, int K = 0) {
  const aom_config& c = a->cfg;
  const int rows = envs ? K : c.n_env;
  NEED(AOM_T_AB, l);
  NEED(AOM_T_STENCIL, l);
  const EnvCond& amp = cond(a, AOM_COND_AMP, l);
  ExtrudeParams p;
  p.screen = a->screen[l]; p.ox = a->ox[l]; p.oy = a->oy[l]; p.count = a->ext_count[l];
  p.k0 = a->in.k0; p.k1 = a->in.k1; p.stencil = (const int*)a->in.tab[AOM_T_STENCIL][l];
  p.N = c.screen_dim[l]; p.S = c.stencil_size[l]; p.E = c.n_env; p.layer = l; p.axis = axis; p.sign = sign;
  p.amp = amp.common; p.amp_env = amp.dev;
  p.ldz = AOM_LD(p.S + p.N); p.Z = a->Z; p.zref = a->zref; p.ldn = AOM_LD(p.N); p.newcol = a->newcol;
  p.steps = steps; p.pass = pass; p.envs = envs;
  if (a->in.opt[AOM_OPT_EXTRUDE_PATH] == AOM_EXTRUDE_I8) {
    // exact integer contraction on tcgen05 (extrude_i8.cuh): digits of the inputs, 13 int8 digit-pair products with
    // int32 accumulators, one rounding to float32 after adding the reference pixel
    const OzOperator& op = a->ab[l];
    const int MT = (rows + OZ_BM - 1) / OZ_BM;
    CU(oz_scratch_reserve(a->oz, MT, op.kb, c.n_env, st));
    OzGatherParams g;
    g.screen = p.screen; g.ox = p.ox; g.oy = p.oy; g.count = p.count; g.k0 = p.k0; g.k1 = p.k1; g.stencil = p.stencil;
    g.zref = p.zref; g.ev = a->oz.ev; g.Zs = a->oz.zs; g.N = p.N; g.S = p.S; g.E = rows; g.KB = op.kb; g.layer = l;
    g.axis = axis; g.sign = sign; g.amp = p.amp; g.amp_env = p.amp_env;
    g.steps = steps; g.pass = pass; g.envs = envs;
    OzGemmParams m;
    m.Zs = a->oz.zs; m.ABs = op.planes; m.ev = a->oz.ev; m.ea = op.ea; m.zref = p.zref;
    m.out = p.newcol; m.ldo = p.ldn; m.E = rows; m.N = p.N; m.KB = op.kb; m.err = a->in.err_word;
    cudaError_t le = oz_extrude_launch(g, m, MT, op.nt, st);
    if (le != cudaSuccess) return report(err, AOM_ERR_CUDA, "oz_extrude_launch: %s", cudaGetErrorString(le));
    *a->in.launches += 2;
    p.zref = nullptr;                                  // the reference pixel is already in the new column
  } else {
    with<false, true>(steps != nullptr, [&](auto PE) { extrude_gather_kernel<PE><<<rows, 256, 0, st>>>(p); });
    KCHECK();
    GemmParams g;
    memset(&g, 0, sizeof(g));
    g.A = a->Z; g.lda = p.ldz; g.B = (const float*)a->in.tab[AOM_T_AB][l]; g.ldb = p.ldz; g.C = a->newcol; g.ldc = p.ldn;
    g.M = rows; g.N = p.N; g.K = p.S + p.N;
    int rc = gemm_launch(g, 0, 1, true, a->in.opt[AOM_OPT_GEMM_PATH], a->in.num_sms, a->in.err_word, st, err);
    if (rc) return rc;
    KCHECK();
  }
  with<false, true>(steps != nullptr, [&](auto PE) { extrude_scatter_kernel<PE><<<rows, EXTRUDE_SCATTER_THREADS, 0, st>>>(p); });
  KCHECK();
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// the wind state
static bool wind_any_env(const Atmos* a) {
  for (int l = 0; l < a->cfg.n_layers; ++l)
    if (cond(a, AOM_COND_WIND_X, l).host || cond(a, AOM_COND_WIND_Y, l).host) return true;
  return false;
}

// The pupil footprint of layer l, with the offsets box (min / max of ix, then of iy), stays on the screen.  The one check
// of it: the samplers read N + 1 pixels from the offset on.
static int footprint(const Atmos* a, int l, const int box[4], char (&err)[512]) {
  const aom_config& c = a->cfg;
  if (box[0] < 0 || box[2] < 0 || box[1] + c.n + 1 > c.screen_dim[l] || box[3] + c.n + 1 > c.screen_dim[l])
    return report(err, AOM_ERR_UNSUPPORTED, "layer %d: pupil footprint leaves the screen", l);
  return AOM_OK;
}

// One transition of the wind state of every layer and environment (wind_host.h) on the device, asynchronously on `st`,
// and the same on the host mirror: passes per layer and offset bounds.  WIND_RESET_ENVS: WIND_RESET of the K
// environments listed in envs_d (device) / envs_h (host) only.  WIND_LOAD_ENVS: their accumulators <- acc_d (device) /
// acc_h (host), both [L][2][K].
static int wind_update(Atmos* a, int mode, cudaStream_t st, char (&err)[512], const int* envs_d = nullptr,
                       const int* envs_h = nullptr, int K = 0, const double* acc_d = nullptr, const double* acc_h = nullptr) {
  const aom_config& c = a->cfg;
  const int E = c.n_env, L = c.n_layers;
  if (L == 0) return AOM_OK;
  WindStateParams P;
  memset(&P, 0, sizeof(P));
  for (int l = 0; l < L; ++l) {
    WindLayerParams& W = P.layer[l];
    const EnvCond &wx = cond(a, AOM_COND_WIND_X, l), &wy = cond(a, AOM_COND_WIND_Y, l);
    W.dx = wx.dev; W.dy = wy.dev; W.cdx = wx.common; W.cdy = wy.common;
    W.ax0 = a->accx[l]; W.ay0 = a->accy[l]; W.xoff = c.wfs_xoff[l]; W.yoff = c.wfs_yoff[l]; W.n2 = 2 * c.screen_dim[l];
  }
  P.acc = a->wind_acc; P.steps = a->wind_steps; P.rec = a->wind_rec; P.E = E; P.n_layers = L; P.mode = mode;
  P.envs = envs_d; P.K = K;
  if (mode == WIND_LOAD_ENVS) {
    WindLoadParams Q;
    memset(&Q, 0, sizeof(Q));
    for (int l = 0; l < L; ++l) { Q.xoff[l] = c.wfs_xoff[l]; Q.yoff[l] = c.wfs_yoff[l]; }
    Q.acc = a->wind_acc; Q.steps = a->wind_steps; Q.rec = a->wind_rec; Q.envs = envs_d; Q.acc_in = acc_d;
    Q.E = E; Q.K = K; Q.n_layers = L;
    wind_load_kernel<<<(L * K + 255) / 256, 256, 0, st>>>(Q);
  } else {
    const int n = mode == WIND_RESET_ENVS ? K : E;
    wind_state_kernel<<<(L * n + 255) / 256, 256, 0, st>>>(P);
  }
  KCHECK();
  for (int l = 0; l < L; ++l) {
    WindLayerParams H = P.layer[l];
    H.dx = cond(a, AOM_COND_WIND_X, l).host; H.dy = cond(a, AOM_COND_WIND_Y, l).host;
    double* ax = a->wind_hacc + (size_t)2 * l * E;
    const double* lx = acc_h ? acc_h + (size_t)2 * l * K : nullptr;
    wind_mirror(mode, H, E, ax, ax + E, envs_h, K, lx, lx ? lx + K : nullptr, a->wind_passes[l], a->wind_box[l]);
  }
  return AOM_OK;
}

// Back to the common accumulators once no layer has winds of its own and every layer's accumulators agree over the batch
// (at the latest after the next aom_reset, which zeroes them): the uniform kernels then run again.
static void wind_try_uniform(Atmos* a) {
  if (!a->wind_pe || wind_any_env(a)) return;
  const int E = a->cfg.n_env;
  for (int l = 0; l < a->cfg.n_layers; ++l) {
    const double* h = a->wind_hacc + (size_t)2 * l * E;
    for (int e = 1; e < E; ++e)
      if (h[e] != h[0] || h[E + e] != h[E]) return;
  }
  for (int l = 0; l < a->cfg.n_layers; ++l) {
    a->accx[l] = a->wind_hacc[(size_t)2 * l * E];
    a->accy[l] = a->wind_hacc[(size_t)(2 * l + 1) * E];
  }
  a->wind_pe = false;
}

// Per-environment wind state from the common one (WIND_INIT on `st`): every environment continues from the layer's
// common accumulators.
static int wind_begin_pe(Atmos* a, cudaStream_t st, char (&err)[512]) {
  const size_t LE = (size_t)a->cfg.n_layers * a->cfg.n_env;
  if (!a->wind_acc) {
    CU(dalloc(&a->wind_acc, 2 * LE));
    CU(dalloc(&a->wind_steps, 2 * LE));
    CU(cudaMalloc((void**)&a->wind_rec, LE * sizeof(WindRec)));
    a->wind_hacc = (double*)calloc(2 * LE, sizeof(double));
    if (!a->wind_hacc) return report(err, AOM_ERR_INVALID, "out of host memory");
  }
  int rc = wind_update(a, WIND_INIT, st, err);
  if (rc) return rc;
  a->wind_pe = true;
  return AOM_OK;
}

int atmos_settle(Atmos* a, int layer, char (&err)[512]) {
  if (!cond(a, AOM_COND_WIND_X, layer).host) {
    wind_try_uniform(a);
    return AOM_OK;
  }
  if (!a->wind_pe) {
    int rc = wind_begin_pe(a, 0, err);
    if (rc) return rc;
    CU(cudaStreamSynchronize(0));                    // the legacy stream: the state is read next on any stream
  }
  return footprint(a, layer, a->wind_box[layer], err);
}

int atmos_move(Atmos* a, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = a->cfg;
  if (a->wind_pe) {
    // per-environment winds: counts and offsets on the device, passes sized by the host mirror (x then y, as below);
    // an environment takes part in the first |count| passes of each axis
    int rc = wind_update(a, WIND_STEP, st, err);
    if (rc) return rc;
    const size_t E = c.n_env;
    for (int l = 0; l < c.n_layers; ++l)
      for (int ax = 0; ax < 2; ++ax)
        for (int i = 0; i < a->wind_passes[l][ax]; ++i) {
          rc = extrude_once(a, l, ax, 1, st, err, a->wind_steps + (2 * l + ax) * E, i);
          if (rc) return rc;
        }
    wind_try_uniform(a);
    return AOM_OK;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    const int nx = wind_advance(a->accx[l], cond(a, AOM_COND_WIND_X, l).common);
    const int ny = wind_advance(a->accy[l], cond(a, AOM_COND_WIND_Y, l).common);
    for (int i = 0; i < abs(nx); ++i) { int rc = extrude_once(a, l, 0, nx > 0 ? 1 : -1, st, err); if (rc) return rc; }
    for (int i = 0; i < abs(ny); ++i) { int rc = extrude_once(a, l, 1, ny > 0 ? 1 : -1, st, err); if (rc) return rc; }
  }
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// Start-up of the screens of every environment (envs null) or of the K environments envs[0..K) (device list, compacted
// extrusions): zero screens, ring origins and counters are expected, and the wind state of WIND_RESET (WIND_RESET_ENVS).
// (The layers' start-up chains are independent, but running them on separate streams with private scratch gained
// nothing for the whole batch -- 1.35 s either way at 4096 environments: every extrusion kernel fills the GPU by itself.)
static int start_screens(Atmos* a, const int* envs, int K, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = a->cfg;
  const size_t E = c.n_env;
  const unsigned rows = envs ? (unsigned)K : (unsigned)E;
  int rc;
  for (int l = 0; l < c.n_layers; ++l) {
    size_t N = c.screen_dim[l];
    int sign = cond(a, AOM_COND_WIND_X, l).common < 0 ? -1 : 1;
    const int* steps = a->wind_pe ? a->wind_steps + (2 * l + 1) * E : nullptr;
    // The reference starts a screen with 2N extrusions along x (columns: 648 pixels in 648 different DRAM rows per
    // environment, the expensive direction of the [y][x] layout -- 0.32 ms per extrusion at 4096 environments against
    // 0.19 ms along y).  From a zero screen with zero ring offsets the recursion along y produces exactly the transpose
    // (same stencil, same operator, same innovation counters; every index expression of the gather / scatter swaps its
    // roles, atmos_kernels.cuh / extrude_i8.cuh), and 2N extrusions bring the ring origin back to zero: so the start-up
    // runs along y and the screens are transposed in place once at the end -- bit-identical pixels, 1.29 -> 0.8 s.
    for (size_t i = 0; i < 2 * N; ++i) { rc = extrude_once(a, l, 1, sign, st, err, steps, (int)i, envs, K); if (rc) return rc; }
    {
      const int T = (int)((N + 31) / 32);
      transpose_screens_kernel<<<dim3((unsigned)(T * (T + 1) / 2), rows), dim3(32, 8), 0, st>>>(a->screen[l], (int)N, envs);
      KCHECK();
      // ring origin: 2N steps along y leave oy = 0 as 2N steps along x leave ox = 0 (2N mod N); nothing to swap
    }
  }
  return AOM_OK;
}

int atmos_reset(Atmos* a, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = a->cfg;
  const size_t E = c.n_env;
  for (int l = 0; l < c.n_layers; ++l) a->accx[l] = a->accy[l] = 0.0;
  if (a->wind_pe && !wind_any_env(a)) a->wind_pe = false;      // every accumulator restarts from 0: common again
  if (a->wind_pe) {
    // per-environment winds: accumulators 0, start-up counts 2N along y signed like each environment's x wind
    int rc = wind_update(a, WIND_RESET, st, err);
    if (rc) return rc;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    size_t N = c.screen_dim[l];
    CU(cudaMemsetAsync(a->screen[l], 0, E * N * N * 4, st));
    CU(cudaMemsetAsync(a->ox[l], 0, E * 4, st));
    CU(cudaMemsetAsync(a->oy[l], 0, E * 4, st));
    CU(cudaMemsetAsync(a->ext_count[l], 0, E * 4, st));
  }
  return start_screens(a, nullptr, 0, st, err);
}

int atmos_reset_envs(Atmos* a, const int* envs_d, const int* envs_h, int K, cudaStream_t st, char (&err)[512]) {
  if (a->cfg.n_layers == 0) return AOM_OK;
  // The listed environments' accumulators restart from 0 while the others keep theirs: the per-environment wind state
  // (common winds included) until they agree again (wind_try_uniform)
  int rc;
  if (!a->wind_pe) { rc = wind_begin_pe(a, st, err); if (rc) return rc; }
  rc = wind_update(a, WIND_RESET_ENVS, st, err, envs_d, envs_h, K);
  if (rc) return rc;
  return start_screens(a, envs_d, K, st, err);
}

int atmos_load(Atmos* a, int n, const int* envs_d, const int* envs_h, const aom_env_head* h, double* stage,
               cudaStream_t st, char (&err)[512]) {
  const int L = a->cfg.n_layers;
  if (L == 0) return AOM_OK;
  // the per-environment state unless the loaded accumulators are the batch's common ones
  bool differ = a->wind_pe;
  for (int k = 0; k < n && !differ; ++k)
    for (int l = 0; l < L; ++l) differ = differ || h[k].acc[l][0] != a->accx[l] || h[k].acc[l][1] != a->accy[l];
  if (!differ) return AOM_OK;
  int rc;
  if (!a->wind_pe) { rc = wind_begin_pe(a, st, err); if (rc) return rc; }
  for (int l = 0; l < L; ++l)
    for (int k = 0; k < n; ++k) {
      stage[(size_t)2 * l * n + k] = h[k].acc[l][0];
      stage[(size_t)(2 * l + 1) * n + k] = h[k].acc[l][1];
    }
  if (!a->snap_acc) CU(dalloc(&a->snap_acc, (size_t)2 * L * a->cfg.n_env));
  CU(cudaMemcpyAsync(a->snap_acc, stage, (size_t)2 * L * n * sizeof(double), cudaMemcpyHostToDevice, st));
  rc = wind_update(a, WIND_LOAD_ENVS, st, err, envs_d, envs_h, n, a->snap_acc, stage);
  if (rc) return rc;
  CU(cudaStreamSynchronize(st));
  for (int l = 0; l < L; ++l) {
    rc = footprint(a, l, a->wind_box[l], err);
    if (rc) return rc;
  }
  wind_try_uniform(a);
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
int atmos_fill_layers(const Atmos* a, WfsParams& p, char (&err)[512]) {
  const aom_config& c = a->cfg;
  for (int l = 0; l < p.n_layers; ++l) {
    WfsLayer& L = p.layer[l];
    L.screen = a->screen[l]; L.ox = a->ox[l]; L.oy = a->oy[l]; L.N = c.screen_dim[l];
    const WindRec r = wind_record(c.wfs_xoff[l], c.wfs_yoff[l], a->accx[l], a->accy[l]);
    L.ix = r.ix; L.iy = r.iy; L.fx = r.fx; L.fy = r.fy; L.w00 = r.w00; L.w01 = r.w01; L.w10 = r.w10; L.w11 = r.w11;
    const int box[4] = {L.ix, L.ix, L.iy, L.iy};    // with per-environment winds: the extremes over the batch
    int rc = footprint(a, l, a->wind_pe ? a->wind_box[l] : box, err);
    if (rc) return rc;
  }
  p.wind = (a->wind_pe && p.n_layers > 0) ? a->wind_rec : nullptr;
  return AOM_OK;
}

const double* atmos_snap_view(const Atmos* a, double (*acc)[2]) {
  for (int l = 0; l < a->cfg.n_layers; ++l) { acc[l][0] = a->accx[l]; acc[l][1] = a->accy[l]; }
  return a->wind_pe ? a->wind_acc : nullptr;
}
