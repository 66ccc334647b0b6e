// libaomarl.so -- C ABI implementation (see include/aomarl.h for the contract and reference citations).
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <algorithm>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/aomarl.h"
#include "dispatch.h"
#include "dalloc.h"
#include "atmos_host.h"
#include "gemm_host.h"
#include "rtc_host.h"
#include "snapshot_kernels.cuh"
#include "pupil_kernels.cuh"
#include "wfs_frame_host.h"
#include "geo_kernels.cuh"
#include "pupil_sweep.cuh"
#include "denoise_kernels.cuh"
#include "denoise_tc_host.h"

static char g_create_error[512] = "";

struct aom_ctx {
  aom_config cfg;
  char err[512];
  int device;
  int num_sms;
  uint64_t launches;
  // tables
  void* tab[AOM_T_COUNT][AOM_MAX_LAYERS];
  size_t tab_bytes[AOM_T_COUNT][AOM_MAX_LAYERS];
  // the turbulence layers: screens, wind state, extrusion (atmos.cu)
  Atmos* atmos;
  uint32_t *k0, *k1;          // device [E] Philox keys (environment seeds)
  // the controller: integrator, RL vectors, actors of every policy slot, per-environment controllers (rtc.cu)
  Rtc* rtc;
  // sensor
  float *slopes_frame, *slopes;
  float *bincube, *phase;
  const float* cube_override;
  double* tar_mom;            // [2][E][5] pupil sums of the target phase (aom_comp_strehl): main target, geometric one
  float* tar_acc;             // [E][TAR_ACC] running sums for the long-exposure figures (SE, variance, 9 core pixels)
  int tar_n;
  // geometric controller (geo_kernels.cuh), allocated on first use
  float *geo_com, *geo_volts, *geo_b, *geo_T, *strehl_geo, *geo_acc;
  double* geo_mom;            // [E][4] pupil sums of m phi, m phi tt_x, m phi tt_y
  int geo_gp, geo_tar_n;
  cudaEvent_t ev_geo;
  // pupil sweep (pupil_sweep.cuh): mask / tip-tilt planes repacked in the lattice frame
  int sweep_state;            // 0 = not prepared, 1 = eligible, -1 = not eligible
  uint32_t* sweep_mask;
  float* sweep_ttp;
  int sweep_nb;               // 128-pixel column blocks per pupil row
  int lds, lda;
  uint32_t frame;
  // the conditions [aom_condition][layer] (layer 0 for those of the sensor and the controller); the only copy of them
  // after aom_create, which clears their initial values in cfg
  EnvCond cond[AOM_COND_COUNT][AOM_MAX_LAYERS];
  int opt[AOM_OPT_COUNT];
  long long* dn_dbg;
  float dn_prm[DT_NPARAM];    // float parameters of the tensor-core denoiser (head of AOM_T_DENOISER_TC)
  int tar_peak, geo_tar_peak; // whether the pending target sums hold the PSF core (AOM_TAR_PEAK)
  int* d_err;                 // device error word raised by bounded waits (gemm_tc.cuh)
  float* strehl;
  uint32_t step;              // the batch's actor decisions (the exploration-noise counter)
  bool seeded;
  // staggered environments (aom_reset_envs): from the first partial reset until the next aom_reset every environment
  // counts its noise frames, actor decisions and long-exposure frames from its own reset, and an environment whose
  // first step is pending (first[e]) takes no action and accumulates no Strehl in its next rl half-step
  bool staggered;
  bool first_any;              // some first[e] may be set (cleared by aom_state_end)
  int* rs_envs;                // device [E] environments of the last aom_reset_envs
  uint32_t* rs_seeds;          // device [2][E] their seeds (low, high words)
  uint32_t* frame0;            // device [E] global noise frame of each environment's first frame
  uint32_t* step_env;          // device [E] actor decision counters
  int* le_n;                   // device [2][E] long-exposure counts (main target, geometric target)
  int* first;                  // device [E] first step pending
  // snapshots (aom_save_envs / aom_load_envs): device list of environments, and the host staging block it is copied
  // from (kept until the stream has passed the copy)
  int* snap_envs;
  void* snap_h;
  size_t snap_h_bytes;
  // the sensor frame's kernel routing and the derived tables of its staged kernels (wfs_frame.cu)
  WfsFrame* wfs;
  // aom_step runs the turbulence update next to the actor / controller GEMMs on a second stream
  cudaStream_t side_stream;
  cudaEvent_t ev_fork, ev_join;
  // device time of the sensor kernel (AOM_OPT_TIME_WFS): event pairs around its launches, read by aom_wfs_time_ms
  cudaEvent_t wev[2][AOM_WFS_TIMERS];
  int wev_n;
};

static int fail(aom_ctx* c, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(c ? c->err : g_create_error, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t _e = (call);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return fail(ctx, AOM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define KCHECK()                                                                                  \
  do {                                                                                            \
    ctx->launches++;                                                                              \
    cudaError_t _e = cudaGetLastError();                                                          \
    if (_e != cudaSuccess)                                                                        \
      return fail(ctx, AOM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

extern "C" size_t aom_config_size(void) { return sizeof(aom_config); }

extern "C" const char* aom_last_error(const aom_ctx* ctx) { return ctx ? ctx->err : g_create_error; }

extern "C" int aom_create(const aom_config* cfg, aom_ctx** out) {
  aom_ctx* ctx = nullptr;
  if (!cfg || !out) return fail(nullptr, AOM_ERR_INVALID, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, AOM_ERR_CUDA, "no CUDA device available: libaomarl has no CPU path");
  if (cfg->n_env < 1 || cfg->n_env > 65535) return fail(nullptr, AOM_ERR_INVALID, "n_env must be in [1, 65535]");
  if (cfg->n_layers < 0 || cfg->n_layers > AOM_MAX_LAYERS) return fail(nullptr, AOM_ERR_INVALID, "n_layers out of range");
  if (cfg->pdiam != 16 || cfg->npix != 16)
    return fail(nullptr, AOM_ERR_UNSUPPORTED, "only pdiam = npix = 16 Shack-Hartmann subapertures are implemented");
  if (!((cfg->nfft == 64 && cfg->nrebin == 2) || (cfg->nfft == 128 && cfg->nrebin == 4)))
    return fail(nullptr, AOM_ERR_UNSUPPORTED, "only (Nfft, nrebin) = (64, 2) or (128, 4) are implemented");
  if (cfg->stamp_size > 64) return fail(nullptr, AOM_ERR_UNSUPPORTED, "actuator stamp larger than 64 pixels");
  if (cfg->pzt_pitch > 0 && (cfg->stamp_size + 15 + cfg->pzt_pitch - 1) / cfg->pzt_pitch + 1 > WFS_NG_MAX)
    return fail(nullptr, AOM_ERR_UNSUPPORTED, "actuator pitch too small for the %d-cell neighbourhood", WFS_NG_MAX);
  if (cfg->delay < 0 || cfg->delay > 2) return fail(nullptr, AOM_ERR_UNSUPPORTED, "controller delay must be 0, 1 or 2 frames");

  ctx = (aom_ctx*)calloc(1, sizeof(aom_ctx));
  if (!ctx) return fail(nullptr, AOM_ERR_INVALID, "out of host memory");
  ctx->cfg = *cfg;
  for (int l = 0; l < AOM_MAX_LAYERS; ++l) {
    ctx->cond[AOM_COND_AMP][l].common = cfg->amp[l];
    ctx->cond[AOM_COND_WIND_X][l].common = cfg->deltax[l];
    ctx->cond[AOM_COND_WIND_Y][l].common = cfg->deltay[l];
    ctx->cfg.amp[l] = ctx->cfg.deltax[l] = ctx->cfg.deltay[l] = 0.f;
  }
  ctx->cond[AOM_COND_NOISE][0].common = cfg->noise;
  ctx->cond[AOM_COND_NPHOTONS][0].common = cfg->nphotons;
  ctx->cond[AOM_COND_GAIN][0].common = cfg->gain;
  ctx->cond[AOM_COND_DELAY][0].common = (float)cfg->delay;
  ctx->cfg.noise = ctx->cfg.nphotons = ctx->cfg.gain = 0.f;
  ctx->cfg.delay = 0;
  ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_UMMA_WS;
  {
    // development overrides of the default kernel paths (see aom_set_option)
    const char* g = getenv("AOM_GEMM_PATH");
    if (g && !strcmp(g, "simt")) ctx->opt[AOM_OPT_GEMM_PATH] = AOM_GEMM_SIMT;
    const char* w = getenv("AOM_WFS_PATH");
    if (w && !strcmp(w, "umma_fast")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_UMMA_FAST;
    if (w && !strcmp(w, "umma")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_UMMA;
    if (w && !strcmp(w, "simt")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_SIMT;
    if (w && !strcmp(w, "tensor_reg")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_MMA_REG;
    if (w && !strcmp(w, "tensor")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_MMA_STAGED;
    if (w && !strcmp(w, "tensor_fast")) ctx->opt[AOM_OPT_WFS_PATH] = AOM_WFS_MMA_STAGED_FAST;
  }
  *out = ctx;   // returned even on failure so that aom_last_error / aom_destroy work
  CU(cudaGetDevice(&ctx->device));
  CU(cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, ctx->device));
  const size_t E = cfg->n_env;
  ctx->lds = AOM_LD(cfg->nslopes);
  ctx->lda = AOM_LD(cfg->nactu);
  CU(dalloc(&ctx->k0, E));
  CU(dalloc(&ctx->k1, E));
  CU(dalloc(&ctx->d_err, 1));
  const AtmosLinks links = {ctx->cond, ctx->tab, ctx->opt, ctx->k0, ctx->k1, ctx->d_err, &ctx->launches, ctx->num_sms};
  int rc = atmos_create(ctx->cfg, links, &ctx->atmos, ctx->err);
  if (rc) return rc;
  CU(dalloc(&ctx->slopes_frame, E * ctx->lds));
  CU(dalloc(&ctx->slopes, E * ctx->lds));
  const RtcLinks rl = {&ctx->cond[AOM_COND_GAIN][0], &ctx->cond[AOM_COND_DELAY][0], ctx->tab, ctx->opt, ctx->k0, ctx->k1, ctx->d_err, &ctx->launches,
                       ctx->num_sms};
  rc = rtc_create(ctx->cfg, rl, &ctx->rtc, ctx->err);
  if (rc) return rc;
  CU(dalloc(&ctx->strehl, E * 4));
  CU(dalloc(&ctx->tar_mom, E * 2 * PSW_MOM2));     // main target, then the geometric controller's
  CU(dalloc(&ctx->tar_acc, E * TAR_ACC));
  CU(cudaMalloc((void**)&ctx->dn_dbg, 32 * sizeof(long long)));
  float* screens[AOM_MAX_LAYERS] = {};
  for (int l = 0; l < cfg->n_layers; ++l) screens[l] = atmos_layer(ctx->atmos, l).screen;
  ctx->wfs = wfs_frame_create(ctx->cfg, screens, ctx->d_err, ctx->num_sms);
  if (!ctx->wfs) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  CU(cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  cudaError_t ae = gemm_init();
  if (ae != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "cudaFuncSetAttribute(dynamic shared memory) failed: %s", cudaGetErrorString(ae));
  return AOM_OK;
}

extern "C" void aom_destroy(aom_ctx* ctx) {
  if (!ctx) return;
  for (int t = 0; t < AOM_T_COUNT; ++t)
    for (int l = 0; l < AOM_MAX_LAYERS; ++l) cudaFree(ctx->tab[t][l]);
  for (int l = 0; l < AOM_MAX_LAYERS; ++l)
    for (int k = 0; k < AOM_COND_COUNT; ++k) { cudaFree(ctx->cond[k][l].dev); free(ctx->cond[k][l].host); }
  atmos_destroy(ctx->atmos);
  rtc_destroy(ctx->rtc);
  void* bufs[] = {ctx->k0, ctx->k1, ctx->slopes_frame, ctx->slopes, ctx->bincube, ctx->phase, ctx->strehl, ctx->tar_mom,
                  ctx->tar_acc, ctx->d_err,
                  ctx->geo_com, ctx->geo_volts, ctx->geo_b, ctx->geo_T, ctx->strehl_geo, ctx->geo_acc, ctx->geo_mom,
                  ctx->sweep_mask, ctx->sweep_ttp, ctx->rs_envs, ctx->rs_seeds, ctx->frame0, ctx->step_env,
                  ctx->le_n, ctx->first, ctx->snap_envs};
  for (void* b : bufs) cudaFree(b);
  wfs_frame_destroy(ctx->wfs);
  for (int i = 0; i < AOM_WFS_TIMERS; ++i)
    for (int j = 0; j < 2; ++j)
      if (ctx->wev[j][i]) cudaEventDestroy(ctx->wev[j][i]);
  if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_geo) cudaEventDestroy(ctx->ev_geo);
  free(ctx->snap_h);
  free(ctx);
}

static size_t table_expected_bytes(const aom_ctx* ctx, int t, int index) {
  const aom_config& c = ctx->cfg;
  const size_t A = c.n_agents;
  switch (t) {
    case AOM_T_AB: return (size_t)c.screen_dim[index] * AOM_LD(c.stencil_size[index] + c.screen_dim[index]) * 4;
    case AOM_T_STENCIL: return (size_t)c.stencil_size[index] * 4;
    case AOM_T_MPUPIL: return (size_t)c.n * c.n * 4;
    case AOM_T_HALFXY: return 256 * 4;
    case AOM_T_SUB_X0: case AOM_T_SUB_Y0: case AOM_T_FLUX: return (size_t)c.nvalid * 4;
    case AOM_T_STAMP1D: return (size_t)c.stamp_size * 4;
    case AOM_T_ACT_MAP: return (size_t)c.pzt_grid_n * c.pzt_grid_n * 4;
    case AOM_T_TT_PLANES: return (size_t)2 * c.tt_dim * c.tt_dim * 4;
    case AOM_T_CMAT: return (size_t)c.nactu * AOM_LD(c.nslopes) * 4;
    case AOM_T_V2M: return (size_t)c.nmodes * AOM_LD(c.nactu) * 4;
    case AOM_T_M2V: return (size_t)c.nactu * AOM_LD(c.nmodes) * 4;
    case AOM_T_FREEDOM: return (size_t)c.nmodes * 4;
    case AOM_T_ACTION_MAP: return (size_t)c.action_dim * 4;
    case AOM_T_STATE_MAP: case AOM_T_NORM_DM_MEAN: case AOM_T_NORM_DM_STD: case AOM_T_NORM_RES_MEAN:
    case AOM_T_NORM_RES_STD: return (size_t)c.state_modes * 4;
    case AOM_T_AGENT_IDX: return A * c.actor_in * 4;
    case AOM_T_AGENT_ACT: return A * c.actor_out * 4;
    case AOM_T_AGENT_REWARD: return A * 2 * 4;
    case AOM_T_ACTOR_W1: return A * c.actor_hidden * AOM_LD(c.actor_in) * 4;
    case AOM_T_ACTOR_B1: case AOM_T_ACTOR_B2: return A * c.actor_hidden * 4;
    case AOM_T_ACTOR_W2: return A * c.actor_hidden * AOM_LD(c.actor_hidden) * 4;
    case AOM_T_ACTOR_WH: return A * 2 * c.actor_out * AOM_LD(c.actor_hidden) * 4;
    case AOM_T_ACTOR_BH: return A * 2 * c.actor_out * 4;
    case AOM_T_GEO_PROJ: return (size_t)c.nactu * AOM_LD(c.nactu) * 4;
    case AOM_T_GEO_SIFN: return (size_t)c.nactu * 4;
    case AOM_T_DENOISER: return (size_t)DN_PARAM_FLOATS * 4;
    case AOM_T_DENOISER_TC: return (size_t)DT_NPARAM * 4 + DT_WBLOB_BYTES;
  }
  return 0;
}

extern "C" int aom_set_table(aom_ctx* ctx, int table, int index, const void* host, size_t nbytes) {
  if (!ctx || !host) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (table < 0 || table >= AOM_T_COUNT || index < 0 || index >= AOM_MAX_LAYERS)
    return fail(ctx, AOM_ERR_INVALID, "table id %d / index %d out of range", table, index);
  size_t want = table_expected_bytes(ctx, table, index);
  if (want != nbytes)
    return fail(ctx, AOM_ERR_INVALID, "Dimension mismatch: table %d[%d] expects %zu bytes, got %zu", table, index, want, nbytes);
  // operators of the integer contraction first: a non-finite one is refused before anything changes
  int rc = atmos_set_table(ctx->atmos, table, index, host, ctx->err);
  if (!rc) rc = rtc_set_table(ctx->rtc, table, index, host, ctx->err);
  if (rc) return rc;
  if (ctx->tab[table][index]) { cudaFree(ctx->tab[table][index]); ctx->tab[table][index] = nullptr; }
  CU(cudaMalloc(&ctx->tab[table][index], nbytes ? nbytes : 4));
  CU(cudaMemcpy(ctx->tab[table][index], host, nbytes, cudaMemcpyHostToDevice));
  ctx->tab_bytes[table][index] = nbytes;
  if (!wfs_frame_set_table(ctx->wfs, table, host, nbytes)) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  if (table == AOM_T_MPUPIL || table == AOM_T_TT_PLANES) ctx->sweep_state = 0;
  if (table == AOM_T_DENOISER_TC) memcpy(ctx->dn_prm, host, (size_t)DT_NPARAM * 4);   // float parameters travel as kernel arguments
  return AOM_OK;
}

#define NEED(t, i)                                                                     \
  do {                                                                                 \
    if (!ctx->tab[t][i]) return fail(ctx, AOM_ERR_STATE, "table %s[%d] not uploaded", #t, i); \
  } while (0)

extern "C" int aom_device_count_launches(const aom_ctx* ctx, uint64_t* n) {
  if (!ctx || !n) return AOM_ERR_INVALID;
  *n = ctx->launches;
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// pupil sweep: eligibility, repacked tables, launch
static int fill_wfs_params(aom_ctx* ctx, WfsParams& p, int flags, float noise);

static int sweep_prepare(aom_ctx* ctx, cudaStream_t st) {
  if (ctx->sweep_state) return AOM_OK;
  const aom_config& c = ctx->cfg;
  ctx->sweep_state = -1;
  const int xs0 = c.pzt_i1_0 - c.pzt_off, ys0 = c.pzt_j1_0 - c.pzt_off;
  if (c.pzt_pitch != 16 || c.stamp_size > 64 || xs0 > 0 || ys0 > 0 || c.n_layers > 4 || !ctx->tab[AOM_T_TT_PLANES][0] ||
      !ctx->tab[AOM_T_STAMP1D][0] || !ctx->tab[AOM_T_ACT_MAP][0])
    return AOM_OK;
  for (int l = 0; l < c.n_layers; ++l)
    if ((c.screen_dim[l] & 3) || c.screen_dim[l] < PSW_BW) return AOM_OK;
  const int nb = (c.n - xs0 + 127) / 128;
  ctx->sweep_nb = nb;
  cudaFree(ctx->sweep_mask); cudaFree(ctx->sweep_ttp);
  ctx->sweep_mask = nullptr; ctx->sweep_ttp = nullptr;
  CU(cudaMalloc((void**)&ctx->sweep_mask, (size_t)c.n * 32 * nb * sizeof(uint32_t)));
  CU(cudaMalloc((void**)&ctx->sweep_ttp, (size_t)2 * c.n * 128 * nb * sizeof(float)));
  WfsParams p;
  int rc = fill_wfs_params(ctx, p, 2, -1.f);
  if (rc) return rc;
  sweep_tables_kernel<<<c.n, 128, 0, st>>>(p, ctx->sweep_mask, ctx->sweep_ttp, nb);
  KCHECK();
  CU(cudaStreamSynchronize(st));     // one-time: later sweeps may run on another stream (aom_step's second stream)
  ctx->sweep_state = 1;
  return AOM_OK;
}

template <int NL, int MODE, bool PE>
static int sweep_launch_t(aom_ctx* ctx, const SweepParams& P, cudaStream_t st) {
  const size_t smem = psw_smem_bytes(NL, PE);
  CU(cudaFuncSetAttribute(pupil_sweep_kernel<NL, MODE, PE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((P.n_strips * P.nb + PSW_WARPS - 1) / PSW_WARPS, P.w.E);
  pupil_sweep_kernel<NL, MODE, PE><<<grid, PSW_WARPS * 32, smem, st>>>(P);
  KCHECK();
  return AOM_OK;
}

// MODE 0: Tp / mom = geometric projection ; MODE 1: mom = pupil sums of m, m phi, m phi^2
template <int MODE>
static int sweep_launch(aom_ctx* ctx, const WfsParams& w, float* Tp, double* mom, cudaStream_t st, float k2t = 0.f,
                        float core_step = 0.f) {
  const aom_config& c = ctx->cfg;
  SweepParams P;
  memset(&P, 0, sizeof(P));
  P.w = w;
  P.maskw = ctx->sweep_mask; P.ttp = ctx->sweep_ttp;
  P.Tp = Tp; P.mom = mom; P.k2t = k2t; P.core_step = core_step;
  P.nb = ctx->sweep_nb;
  P.n_strips = (c.n + PSW_STRIP - 1) / PSW_STRIP;
  P.err = ctx->d_err;
  int rc = AOM_OK;
  // no layer runs as one, more than three as four
  with<1, 2, 3, 4>(std::min(std::max(w.n_layers, 1), 4), [&](auto NL) {
    with<false, true>(w.wind != nullptr, [&](auto PE) { rc = sweep_launch_t<NL, MODE, PE>(ctx, P, st); });
  });
  return rc;
}

// buffers of the geometric controller (only configurations that use it pay for them)
static int geo_prepare(aom_ctx* ctx) {
  if (ctx->geo_com) return AOM_OK;
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  if (c.pzt_grid_n < 1 || c.pzt_pitch < 1) return fail(ctx, AOM_ERR_UNSUPPORTED, "geometric controller needs the actuator lattice");
  ctx->geo_gp = AOM_LD(c.pzt_grid_n);
  CU(dalloc(&ctx->geo_volts, E * ctx->lda));
  CU(dalloc(&ctx->geo_b, E * ctx->lda));
  {
    // lattice-column sums of every pupil row: [E][n][gp], or the sweep's per-block partials [E][n][nb][PSW_TP]
    const int xs0 = c.pzt_i1_0 - c.pzt_off;
    const size_t nb = xs0 <= 0 ? (size_t)(c.n - xs0 + 127) / 128 : 0;
    const size_t per_row = nb * PSW_TP > (size_t)ctx->geo_gp ? nb * PSW_TP : (size_t)ctx->geo_gp;
    CU(dalloc(&ctx->geo_T, E * c.n * per_row));
  }
  CU(dalloc(&ctx->geo_mom, E * 4));
  CU(dalloc(&ctx->strehl_geo, E * 4));
  CU(dalloc(&ctx->geo_acc, E * TAR_ACC));
  CU(cudaEventCreateWithFlags(&ctx->ev_geo, cudaEventDisableTiming));
  CU(dalloc(&ctx->geo_com, E * ctx->lda));
  return AOM_OK;
}

extern "C" int aom_get_buffer(aom_ctx* ctx, int buffer, int index, void** dptr, size_t* count) {
  if (!ctx || !dptr || !count) return fail(ctx, AOM_ERR_INVALID, "null argument");
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  const RtcView v = rtc_view(ctx->rtc);
  void* p = nullptr;
  size_t n = 0;
  switch (buffer) {
    case AOM_B_SCREEN:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = atmos_layer(ctx->atmos, index).screen; n = E * c.screen_dim[index] * c.screen_dim[index]; break;
    case AOM_B_RING_OX:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = atmos_layer(ctx->atmos, index).ox; n = E; break;
    case AOM_B_RING_OY:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = atmos_layer(ctx->atmos, index).oy; n = E; break;
    case AOM_B_EXT_COUNT:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = atmos_layer(ctx->atmos, index).count; n = E; break;
    case AOM_B_SLOPES: p = ctx->slopes; n = E * ctx->lds; break;
    case AOM_B_ERR: p = v.err; n = E * v.lda; break;
    case AOM_B_COM: p = v.com; n = E * v.lda; break;
    case AOM_B_VOLTS: p = v.volts; n = E * v.lda; break;
    case AOM_B_BINCUBE:
      if (!ctx->bincube) CU(dalloc(&ctx->bincube, E * c.nvalid * 256));
      p = ctx->bincube; n = E * c.nvalid * 256; break;
    case AOM_B_PHASE:
      if (!ctx->phase) CU(dalloc(&ctx->phase, E * c.n * c.n));
      p = ctx->phase; n = E * c.n * c.n; break;
    case AOM_B_MODES: p = v.modes; n = E * v.ldm; break;
    case AOM_B_RES_MODES: p = v.modes_res; n = E * v.ldm; break;
    case AOM_B_STATE: p = v.state; n = E * v.ldst; break;
    case AOM_B_REWARD: p = v.reward; n = E * c.n_agents; break;
    case AOM_B_ACTION: p = v.action; n = E * v.ldact; break;
    case AOM_B_ACTION_MEAN: p = v.action_mean; n = E * v.ldact; break;
    case AOM_B_STREHL: p = ctx->strehl; n = E * 4; break;
    case AOM_B_GEO_COM: case AOM_B_GEO_VOLTS: case AOM_B_STREHL_GEO: case AOM_B_GEO_PROJ: {
      int rc = geo_prepare(ctx);
      if (rc) return rc;
      if (buffer == AOM_B_STREHL_GEO) { p = ctx->strehl_geo; n = E * 4; }
      else { p = buffer == AOM_B_GEO_COM ? ctx->geo_com : buffer == AOM_B_GEO_VOLTS ? ctx->geo_volts : ctx->geo_b; n = E * ctx->lda; }
      break;
    }
    default: return fail(ctx, AOM_ERR_INVALID, "unknown buffer id %d", buffer);
  }
  if (!p) return fail(ctx, AOM_ERR_STATE, "buffer %d is not allocated for this configuration", buffer);
  *dptr = p;
  *count = n;
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
extern "C" int aom_gemm_tn(aom_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                           int M, int N, int K, const float* bias, int relu, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.bias = bias; p.relu = relu;
  int rc = gemm_launch(p, 0, 1, false, ctx->opt[AOM_OPT_GEMM_PATH], ctx->num_sms, ctx->d_err, (cudaStream_t)stream, ctx->err);
  if (rc) return rc;
  KCHECK();
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// the conditions (aom_condition)
static const char* const cond_names[AOM_COND_COUNT] = {"amplitude", "wind x", "wind y", "sensor noise", "photon count", "gain",
                                                       "", "delay"};
static_assert(AOM_COND_COUNT == 8, "cond_names and cond_layers list every condition");

// Whether value v is allowed for condition k: finite, photon counts > 0, delays in [0, 2] frames
static const char* cond_refusal(int k, float v) {
  if (!isfinite(v)) return "is not finite";
  if (k == AOM_COND_NPHOTONS && !(v > 0.f)) return "must be > 0";
  if (k == AOM_COND_DELAY && !(v >= 0.f && v <= 2.f)) return "must be in [0, 2] frames";
  return nullptr;
}

// One change of condition (k, l): env false sets the common value *v; env true sets the per-environment values v[E]
// (host), or with v null returns to the common value.
struct CondSet {
  int k, l;
  bool env;
  const float* v;
};

// The one setter of the conditions.  Checks every value of the n changes first (cond_refusal), then
// allocates the arrays of those that become per-environment, all or none: a refused call changes nothing.  Waits for the
// device when per-environment values change (a kernel in flight may still read the old ones).
static int set_conditions(aom_ctx* ctx, int n, const CondSet* s) {
  if (!ctx) return AOM_ERR_INVALID;
  const int E = ctx->cfg.n_env;
  bool env = false;
  for (int i = 0; i < n; ++i) {
    const CondSet& c = s[i];
    if (c.l < 0 || c.l >= cond_layers(c.k, ctx->cfg.n_layers)) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
    env = env || c.env;
    for (int e = 0; e < (!c.v ? 0 : c.env ? E : 1); ++e) {
      const char* why = cond_refusal(c.k, c.v[e]);
      if (!why) continue;
      char where[32] = "", who[32] = "";
      if (c.k <= AOM_COND_WIND_Y) snprintf(where, sizeof(where), "layer %d: ", c.l);
      if (c.env) snprintf(who, sizeof(who), " of environment %d", e);
      return fail(ctx, AOM_ERR_INVALID, "%s%s%s %s", where, cond_names[c.k], who, why);
    }
  }
  if (env) CU(cudaDeviceSynchronize());
  bool fresh[AOM_COND_COUNT * AOM_MAX_LAYERS] = {}, ok = true;
  for (int i = 0; i < n && ok; ++i) {
    EnvCond& C = ctx->cond[s[i].k][s[i].l];
    if (!(fresh[i] = s[i].env && s[i].v && !C.host)) continue;
    C.host = (float*)malloc((size_t)E * sizeof(float));
    ok = C.host && cudaMalloc((void**)&C.dev, (size_t)E * sizeof(float)) == cudaSuccess;
  }
  for (int i = 0; i < n && !ok; ++i)
    if (fresh[i]) { EnvCond& C = ctx->cond[s[i].k][s[i].l]; free(C.host); cudaFree(C.dev); C.host = C.dev = nullptr; }
  if (!ok) return fail(ctx, AOM_ERR_CUDA, "out of memory for per-environment values");
  for (int i = 0; i < n; ++i) {
    EnvCond& C = ctx->cond[s[i].k][s[i].l];
    if (!s[i].env) {
      C.common = *s[i].v;
    } else if (!s[i].v) {
      cudaFree(C.dev); free(C.host);
      C.dev = C.host = nullptr;
    } else {
      CU(cudaMemcpy(C.dev, s[i].v, (size_t)E * sizeof(float), cudaMemcpyHostToDevice));
      memcpy(C.host, s[i].v, (size_t)E * sizeof(float));
    }
  }
  return AOM_OK;
}

extern "C" int aom_get_condition(aom_ctx* ctx, int cond, int layer, float* common, float* values_host, int* per_env) {
  if (!ctx) return AOM_ERR_INVALID;
  if (cond < 0 || cond >= AOM_COND_COUNT || !cond_layers(cond, 1)) return fail(ctx, AOM_ERR_INVALID, "unknown condition %d", cond);
  if (layer < 0 || layer >= cond_layers(cond, ctx->cfg.n_layers)) return fail(ctx, AOM_ERR_INVALID, "%s: layer %d out of range", cond_names[cond], layer);
  const EnvCond& C = ctx->cond[cond][layer];
  if (common) *common = C.common;
  if (per_env) *per_env = C.host != nullptr;
  for (int e = 0; values_host && e < ctx->cfg.n_env; ++e) values_host[e] = C.at(e);
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
extern "C" int aom_set_layer_wind(aom_ctx* ctx, int layer, const float* deltax_host, const float* deltay_host) {
  if (!deltax_host != !deltay_host) return fail(ctx, AOM_ERR_INVALID, "per-environment winds need both components (or neither)");
  const CondSet s[2] = {{AOM_COND_WIND_X, layer, true, deltax_host}, {AOM_COND_WIND_Y, layer, true, deltay_host}};
  int rc = set_conditions(ctx, 2, s);
  return rc ? rc : atmos_settle(ctx->atmos, layer, ctx->err);
}

extern "C" int aom_move_atmos(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_move_atmos");
  return atmos_move(ctx->atmos, (cudaStream_t)stream, ctx->err);
}

static int clear_loop_state(aom_ctx* ctx, cudaStream_t st) {
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  CU(cudaMemsetAsync(ctx->slopes, 0, E * ctx->lds * 4, st));
  CU(cudaMemsetAsync(ctx->slopes_frame, 0, E * ctx->lds * 4, st));
  int rc = rtc_clear(ctx->rtc, st, ctx->err);
  if (rc) return rc;
  ctx->cube_override = nullptr;
  ctx->tar_n = 0;
  CU(cudaMemsetAsync(ctx->tar_acc, 0, E * TAR_ACC * sizeof(float), st));
  CU(cudaMemsetAsync(ctx->strehl, 0, E * 4 * sizeof(float), st));
  if (ctx->geo_com) {
    ctx->geo_tar_n = 0;
    CU(cudaMemsetAsync(ctx->geo_com, 0, E * ctx->lda * 4, st));
    CU(cudaMemsetAsync(ctx->geo_volts, 0, E * ctx->lda * 4, st));
    CU(cudaMemsetAsync(ctx->geo_acc, 0, E * TAR_ACC * sizeof(float), st));
    CU(cudaMemsetAsync(ctx->strehl_geo, 0, E * 4 * sizeof(float), st));
  }
  return AOM_OK;
}

static int stagger_begin(aom_ctx* ctx, cudaStream_t st);

extern "C" int aom_reset(aom_ctx* ctx, const int64_t* seeds, void* stream) {
  if (!ctx || !seeds) return fail(ctx, AOM_ERR_INVALID, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  uint32_t* h = (uint32_t*)malloc(2 * E * sizeof(uint32_t));
  for (size_t e = 0; e < E; ++e) {
    uint64_t s = (uint64_t)seeds[e];
    h[e] = (uint32_t)(s & 0xffffffffu);
    h[E + e] = (uint32_t)(s >> 32);
  }
  cudaError_t e1 = cudaMemcpyAsync(ctx->k0, h, E * 4, cudaMemcpyHostToDevice, st);
  cudaError_t e2 = cudaMemcpyAsync(ctx->k1, h + E, E * 4, cudaMemcpyHostToDevice, st);
  cudaError_t e3 = cudaStreamSynchronize(st);
  free(h);
  CU(e1); CU(e2); CU(e3);
  ctx->seeded = true;
  ctx->frame = 0;
  ctx->step = 0;
  int rc = clear_loop_state(ctx, st);
  if (rc) return rc;
  ctx->staggered = false;                                                // every environment in lockstep again
  ctx->first_any = false;
  if (ctx->first) {
    CU(cudaMemsetAsync(ctx->frame0, 0, E * sizeof(uint32_t), st));
    CU(cudaMemsetAsync(ctx->step_env, 0, E * sizeof(uint32_t), st));
    CU(cudaMemsetAsync(ctx->le_n, 0, 2 * E * sizeof(int), st));
    CU(cudaMemsetAsync(ctx->first, 0, E * sizeof(int), st));
  }
  if (rtc_integrators(ctx->rtc)) {                                       // integrator environments freeze their counters
    rc = stagger_begin(ctx, st);
    if (rc) return rc;
  }
  return atmos_reset(ctx->atmos, st, ctx->err);
}

// Checks a host list of n environments of the batch: n >= 0, every index in range and listed once.
static int check_env_list(aom_ctx* ctx, int n, const int32_t* envs, const char* what) {
  const int E = ctx->cfg.n_env;
  if (n < 0) return fail(ctx, AOM_ERR_INVALID, "%s: negative environment count %d", what, n);
  if (n > 0 && !envs) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (n > E) return fail(ctx, AOM_ERR_INVALID, "%s: %d environments listed, the batch has %d", what, n, E);
  char* seen = (char*)calloc((size_t)E, 1);
  if (!seen) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  for (int k = 0; k < n; ++k) {
    const int e = envs[k];
    if (e < 0 || e >= E) { free(seen); return fail(ctx, AOM_ERR_INVALID, "%s: environment %d out of range [0, %d)", what, e, E); }
    if (seen[e]) { free(seen); return fail(ctx, AOM_ERR_INVALID, "%s: environment %d listed twice", what, e); }
    seen[e] = 1;
  }
  free(seen);
  return AOM_OK;
}

// The batch leaves lockstep (aom_reset_envs, aom_load_envs): per-environment counters, every one at the batch's counts.
static int stagger_begin(aom_ctx* ctx, cudaStream_t st) {
  const int E = ctx->cfg.n_env;
  if (!ctx->first) {
    CU(dalloc(&ctx->rs_envs, (size_t)E));
    CU(dalloc(&ctx->rs_seeds, 2 * (size_t)E));
    CU(dalloc(&ctx->frame0, (size_t)E));
    CU(dalloc(&ctx->step_env, (size_t)E));
    CU(dalloc(&ctx->le_n, 2 * (size_t)E));
    CU(dalloc(&ctx->first, (size_t)E));
  }
  if (!ctx->staggered) {
    stagger_counters_kernel<<<(E + 255) / 256, 256, 0, st>>>(ctx->frame0, ctx->step_env, ctx->le_n, ctx->first, E, ctx->step,
                                                             ctx->tar_n, ctx->geo_tar_n);
    KCHECK();
    ctx->staggered = true;
  }
  return AOM_OK;
}

// The one enumeration of the per-environment rows of the context: word (s * slot_stride + e * ld + i) of buf for s <
// slots, i < ld belongs to environment e.  aom_reset_envs clears the rows marked `clear`; aom_save_envs / aom_load_envs
// pack and unpack all of them.  The others are the Philox keys (aom_reset_envs sets them from the new seeds) and the
// pending target sums (a fresh trace overwrites them).  Buffers not allocated are skipped.
struct EnvRow {
  void* buf;
  long long ld, slot_stride;
  int slots, ring, clear;
};

static int env_rows(const aom_ctx* ctx, EnvRow* out) {
  const aom_config& c = ctx->cfg;
  const long long E = c.n_env;
  const RtcView v = rtc_view(ctx->rtc);
  int n = 0;
  auto add = [&](void* b, long long ld, int clear = 1, int slots = 1, long long slot_stride = 0, int ring = 0) {
    if (b) out[n++] = EnvRow{b, ld, slot_stride, slots, ring, clear};
  };
  add(ctx->slopes, ctx->lds); add(ctx->slopes_frame, ctx->lds); add(v.err, v.lda); add(v.com, v.lda);
  add(v.com1, v.lda); add(v.com2, v.lda); add(v.volts, v.lda); add(v.com_before, v.lda); add(v.modes_res, v.ldm);
  add(v.state, v.ldst); add(v.action, v.ldact); add(ctx->tar_acc, TAR_ACC); add(ctx->strehl, 4);
  add(v.hist, c.state_modes, 1, c.n_hist, E * c.state_modes, 1);         // every slot of the ring
  add(ctx->geo_com, ctx->lda); add(ctx->geo_volts, ctx->lda); add(ctx->geo_acc, TAR_ACC); add(ctx->strehl_geo, 4);
  for (int l = 0; l < c.n_layers; ++l) {
    const AtmosLayer a = atmos_layer(ctx->atmos, l);
    add(a.screen, (long long)c.screen_dim[l] * c.screen_dim[l]);
    add(a.ox, 1); add(a.oy, 1); add(a.count, 1);
  }
  add(ctx->k0, 1, 0); add(ctx->k1, 1, 0);
  add(ctx->tar_mom, 2 * PSW_MOM2, 0, 2, E * 2 * PSW_MOM2);                // doubles [2][E][PSW_MOM2]: both targets
  add(ctx->geo_mom, 2 * 4, 0);                                           // doubles [E][4]
  return n;
}

extern "C" int aom_reset_envs(aom_ctx* ctx, int n, const int32_t* envs, const int64_t* seeds, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  const int E = c.n_env;
  int rc = check_env_list(ctx, n, envs, "aom_reset_envs");
  if (rc) return rc;
  if (n > 0 && !seeds) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_reset_envs");
  if (n == 0) return AOM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CU(cudaStreamSynchronize(st));                     // the wind mirror and the staging buffers are updated from the host
  rc = stagger_begin(ctx, st);
  if (rc) return rc;
  {
    uint32_t* h = (uint32_t*)malloc(2 * (size_t)n * sizeof(uint32_t));
    if (!h) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    for (int k = 0; k < n; ++k) {
      const uint64_t sd = (uint64_t)seeds[k];
      h[k] = (uint32_t)(sd & 0xffffffffu);
      h[n + k] = (uint32_t)(sd >> 32);
    }
    cudaError_t e1 = cudaMemcpyAsync(ctx->rs_envs, envs, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st);
    cudaError_t e2 = cudaMemcpyAsync(ctx->rs_seeds, h, 2 * (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
    cudaError_t e3 = cudaStreamSynchronize(st);
    free(h);
    CU(e1); CU(e2); CU(e3);
  }
  // every per-environment row aom_reset clears, the listed environments' screens and ring state, keys and counters
  ResetEnvsParams P;
  memset(&P, 0, sizeof(P));
  EnvRow rows[SNAP_MAX_SEGS];
  const int nrows = env_rows(ctx, rows);
  for (int i = 0; i < nrows && P.nbuf < RESET_MAX_BUFS; ++i) {
    const EnvRow& r = rows[i];
    if (!r.clear) continue;
    P.buf[P.nbuf] = (uint32_t*)r.buf; P.ld[P.nbuf] = r.ld; P.slots[P.nbuf] = r.slots; P.slot_stride[P.nbuf] = r.slot_stride;
    P.nbuf++;
  }
  P.envs = ctx->rs_envs; P.seeds = ctx->rs_seeds; P.K = n; P.E = E;
  P.k0 = ctx->k0; P.k1 = ctx->k1; P.frame0 = ctx->frame0; P.step_env = ctx->step_env; P.le_n = ctx->le_n;
  P.first = ctx->first; P.frame = ctx->frame;
  reset_envs_kernel<<<dim3((unsigned)n, (unsigned)P.nbuf + 1), 256, 0, st>>>(P);
  KCHECK();
  ctx->first_any = true;
  return atmos_reset_envs(ctx->atmos, ctx->rs_envs, envs, n, st, ctx->err);
}

// ---------------------------------------------------------------------------------------------
// per-environment snapshots (snapshot_kernels.cuh)

// FNV-1a of the configuration without the batch size (the conditions are cleared in ctx->cfg): two contexts whose
// records are interchangeable have the same fingerprint
static uint64_t config_fingerprint(const aom_config& cfg) {
  aom_config c = cfg;
  c.n_env = 0;
  uint64_t h = 1469598103934665603ull;
  const unsigned char* b = (const unsigned char*)&c;
  for (size_t i = 0; i < sizeof(c); ++i) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}

// Segment table of a record (the rows of env_rows after the head) and its size
static size_t snap_layout(const aom_ctx* ctx, SnapParams& P) {
  EnvRow rows[SNAP_MAX_SEGS];
  const int nrows = env_rows(ctx, rows);
  long long off = SNAP_HEAD_BYTES;
  int chunks = 0;
  P.nseg = nrows;
  for (int i = 0; i < nrows; ++i) {
    const EnvRow& r = rows[i];
    SnapSeg& G = P.seg[i];
    G.buf = (uint32_t*)r.buf; G.ld = r.ld; G.slot_stride = r.slot_stride; G.slots = r.slots; G.ring = r.ring;
    G.off = off; G.pitch = (r.ld * 4 + 15) / 16 * 16;
    G.cps = (int)((r.ld + SNAP_CHUNK_WORDS - 1) / SNAP_CHUNK_WORDS);
    G.chunk0 = chunks;
    chunks += G.cps * r.slots;
    off += G.pitch * r.slots;
  }
  P.nchunks = chunks;
  return (size_t)off;
}

extern "C" int aom_env_state_bytes(aom_ctx* ctx, size_t* bytes) {
  if (!ctx || !bytes) return fail(ctx, AOM_ERR_INVALID, "null argument");
  SnapParams P;
  *bytes = snap_layout(ctx, P);
  return AOM_OK;
}

// The parameters of a pack / unpack of n records at rec whose device list of environments is ctx->snap_envs
static void snap_params(aom_ctx* ctx, SnapParams& P, int n, void* rec) {
  const aom_config& c = ctx->cfg;
  memset(&P, 0, sizeof(P));
  const size_t bytes = snap_layout(ctx, P);
  P.envs = ctx->snap_envs; P.rec = (unsigned char*)rec; P.bytes = (long long)bytes;
  P.E = c.n_env; P.hist_head = rtc_view(ctx->rtc).hist_head;
  P.magic = AOM_ENV_MAGIC; P.rec_bytes = (uint32_t)bytes; P.fingerprint = config_fingerprint(c); P.n_layers = c.n_layers;
  P.frame = ctx->frame; P.step = ctx->step; P.le_c[0] = ctx->tar_n; P.le_c[1] = ctx->geo_tar_n;
  if (ctx->staggered) { P.frame0 = ctx->frame0; P.step_env = ctx->step_env; P.le_n = ctx->le_n; P.first = ctx->first; }
  P.wind_acc = atmos_snap_view(ctx->atmos, P.acc_c);
  for (int k = 0; k < AOM_COND_COUNT; ++k)
    for (int l = 0; l < AOM_MAX_LAYERS; ++l) { P.cond_env[k][l] = ctx->cond[k][l].dev; P.cond_c[k][l] = ctx->cond[k][l].common; }
}

// Host staging block of at least `bytes`, and the device list of environments envs[0..n) copied from it on `st`
static int snap_stage(aom_ctx* ctx, int n, const int32_t* envs, size_t bytes, cudaStream_t st) {
  if (!ctx->snap_envs) CU(dalloc(&ctx->snap_envs, (size_t)ctx->cfg.n_env));
  if (bytes < (size_t)n * sizeof(int32_t)) bytes = (size_t)n * sizeof(int32_t);
  if (bytes > ctx->snap_h_bytes) {
    free(ctx->snap_h);
    ctx->snap_h = malloc(bytes);
    ctx->snap_h_bytes = ctx->snap_h ? bytes : 0;
    if (!ctx->snap_h) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  }
  memcpy(ctx->snap_h, envs, (size_t)n * sizeof(int32_t));
  CU(cudaMemcpyAsync(ctx->snap_envs, ctx->snap_h, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  return AOM_OK;
}

extern "C" int aom_save_envs(aom_ctx* ctx, int n, const int32_t* envs, void* dst, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc = check_env_list(ctx, n, envs, "aom_save_envs");
  if (rc) return rc;
  if (n > 0 && !dst) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_save_envs");
  if (n == 0) return AOM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CU(cudaStreamSynchronize(st));                     // the staging block is free and the host mirrors are current
  rc = snap_stage(ctx, n, envs, 0, st);
  if (rc) return rc;
  SnapParams P;
  snap_params(ctx, P, n, dst);
  env_pack_kernel<<<dim3((unsigned)P.nchunks + 1, (unsigned)n), SNAP_THREADS, 0, st>>>(P);
  KCHECK();
  CU(cudaStreamSynchronize(st));
  return AOM_OK;
}

// The conditions of the loaded records: each environment keeps its value in force except envs[k], which takes that of
// record k.  A condition where one of them differs becomes per-environment (a wind both components of its layer), all
// in one set_conditions call: refused values change nothing.
static int load_conditions(aom_ctx* ctx, int n, const int32_t* envs, aom_env_head* h) {
  const int E = ctx->cfg.n_env, L = ctx->cfg.n_layers;
  float* a = (float*)malloc((size_t)AOM_COND_COUNT * AOM_MAX_LAYERS * E * sizeof(float));
  if (!a) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  bool differ[AOM_COND_COUNT][AOM_MAX_LAYERS] = {};
  for (int k = 0; k < AOM_COND_COUNT; ++k)
    for (int l = 0; l < cond_layers(k, L); ++l) {
      float* v = a + (size_t)(k * AOM_MAX_LAYERS + l) * E;
      for (int e = 0; e < E; ++e) v[e] = ctx->cond[k][l].at(e);
      for (int i = 0; i < n; ++i) {
        const float x = head_cond(h[i], k, l);
        differ[k][l] = differ[k][l] || memcmp(&x, &v[envs[i]], sizeof(float)) != 0;
        v[envs[i]] = x;
      }
    }
  for (int l = 0; l < L; ++l)
    differ[AOM_COND_WIND_X][l] = differ[AOM_COND_WIND_Y][l] = differ[AOM_COND_WIND_X][l] || differ[AOM_COND_WIND_Y][l];
  CondSet s[AOM_COND_COUNT * AOM_MAX_LAYERS];
  int ns = 0;
  for (int k = 0; k < AOM_COND_COUNT; ++k)
    for (int l = 0; l < cond_layers(k, L); ++l)
      if (differ[k][l]) s[ns++] = CondSet{k, l, true, a + (size_t)(k * AOM_MAX_LAYERS + l) * E};
  int rc = set_conditions(ctx, ns, s);
  free(a);
  for (int l = 0; l < L && !rc; ++l)
    if (differ[AOM_COND_WIND_X][l]) rc = atmos_settle(ctx->atmos, l, ctx->err);
  return rc;
}

extern "C" int aom_load_envs(aom_ctx* ctx, int n, const int32_t* envs, const void* src, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  const int L = c.n_layers;
  int rc = check_env_list(ctx, n, envs, "aom_load_envs");
  if (rc) return rc;
  if (n > 0 && !src) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_load_envs");
  if (n == 0) return AOM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CU(cudaStreamSynchronize(st));
  // the heads first, checked before anything changes
  size_t bytes;
  aom_env_state_bytes(ctx, &bytes);
  const size_t hs = sizeof(aom_env_head);
  // staging block: the list of environments, then (16-byte aligned) the heads, then the loaded accumulators [L][2][n]
  const size_t at = ((size_t)n * sizeof(int32_t) + 15) / 16 * 16;
  rc = snap_stage(ctx, n, envs, at + (size_t)n * (hs + 2 * L * sizeof(double)), st);
  if (rc) return rc;
  aom_env_head* h = (aom_env_head*)((char*)ctx->snap_h + at);
  CU(cudaMemcpy2DAsync(h, hs, src, bytes, hs, (size_t)n, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const uint64_t fp = config_fingerprint(c);
  for (int k = 0; k < n; ++k) {
    if (h[k].magic != AOM_ENV_MAGIC) return fail(ctx, AOM_ERR_INVALID, "aom_load_envs: record %d is not an environment record", k);
    if (h[k].bytes != bytes || h[k].fingerprint != fp || h[k].n_layers != L)
      return fail(ctx, AOM_ERR_INVALID, "aom_load_envs: record %d (%u bytes) was saved by a context of another configuration or "
                  "allocation (this one: %zu bytes)", k, h[k].bytes, bytes);
  }
  rc = load_conditions(ctx, n, envs, h);
  if (rc) return rc;
  rc = stagger_begin(ctx, st);
  if (rc) return rc;
  SnapParams P;
  snap_params(ctx, P, n, (void*)src);
  env_unpack_kernel<<<dim3((unsigned)P.nchunks + 1, (unsigned)n), SNAP_THREADS, 0, st>>>(P);
  KCHECK();
  ctx->first_any = true;                             // a loaded environment may have its first step pending
  rc = atmos_load(ctx->atmos, n, ctx->snap_envs, envs, h, (double*)(h + n), st, ctx->err);
  if (rc) return rc;
  CU(cudaStreamSynchronize(st));
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// per-environment controllers

extern "C" int aom_set_controller_env(aom_ctx* ctx, const int32_t* ctrl) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc = rtc_set_controller(ctx->rtc, ctrl, ctx->err);
  if (rc || !rtc_integrators(ctx->rtc)) return rc;
  rc = stagger_begin(ctx, nullptr);                  // integrator environments freeze their decision counters
  if (rc) return rc;
  CU(cudaDeviceSynchronize());
  return AOM_OK;
}

extern "C" int aom_get_controller_env(aom_ctx* ctx, int32_t* ctrl, int* per_env) {
  if (!ctx) return AOM_ERR_INVALID;
  rtc_get_controller(ctx->rtc, ctrl, per_env);
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
static int fill_wfs_params(aom_ctx* ctx, WfsParams& p, int flags, float noise) {
  const aom_config& c = ctx->cfg;
  memset(&p, 0, sizeof(p));
  NEED(AOM_T_MPUPIL, 0); NEED(AOM_T_HALFXY, 0); NEED(AOM_T_SUB_X0, 0); NEED(AOM_T_SUB_Y0, 0); NEED(AOM_T_FLUX, 0);
  p.n_layers = (flags & 1) ? c.n_layers : 0;
  int rc = atmos_fill_layers(ctx->atmos, p, ctx->err);
  if (rc) return rc;
  p.use_dm = (flags & 2) ? 1 : 0;
  if (p.use_dm) {
    NEED(AOM_T_STAMP1D, 0); NEED(AOM_T_ACT_MAP, 0); NEED(AOM_T_TT_PLANES, 0);
  }
  p.E = c.n_env; p.n = c.n; p.nvalid = c.nvalid;
  p.mpupil = (const float*)ctx->tab[AOM_T_MPUPIL][0];
  p.halfxy = (const float*)ctx->tab[AOM_T_HALFXY][0];
  p.sub_x0 = (const int*)ctx->tab[AOM_T_SUB_X0][0];
  p.sub_y0 = (const int*)ctx->tab[AOM_T_SUB_Y0][0];
  p.flux = (const float*)ctx->tab[AOM_T_FLUX][0];
  p.volts = rtc_view(ctx->rtc).volts; p.ldv = ctx->lda;
  p.stamp1d = (const float*)ctx->tab[AOM_T_STAMP1D][0]; p.ss = c.stamp_size;
  p.act_map = (const int*)ctx->tab[AOM_T_ACT_MAP][0];
  p.grid_n = c.pzt_grid_n; p.pitch = c.pzt_pitch; p.i1_0 = c.pzt_i1_0; p.j1_0 = c.pzt_j1_0;
  p.pzt_off = c.pzt_off; p.pzt_nact = c.pzt_nact;
  p.tt_planes = (const float*)ctx->tab[AOM_T_TT_PLANES][0]; p.tt_dim = c.tt_dim; p.tt_off = c.tt_off;
  p.k2 = (float)(2.0 * M_PI / (double)c.lambda_um);
  p.nphotons = ctx->cond[AOM_COND_NPHOTONS][0].common; p.noise = noise; p.cog_offset = c.cog_offset; p.pixsize = c.pixsize;
  // per-environment sensor values: every frame is scaled by each environment's photon count, a noisy frame (noise >= 0)
  // draws each environment's own noise, a noise-free one none
  p.nph_env = ctx->cond[AOM_COND_NPHOTONS][0].dev;
  p.noise_env = (noise >= 0.f) ? ctx->cond[AOM_COND_NOISE][0].dev : nullptr;
  p.frame = ctx->frame; p.wfs_index = (uint32_t)c.wfs_index; p.k0 = ctx->k0; p.k1 = ctx->k1;
  p.frame0 = ctx->staggered ? ctx->frame0 : nullptr;
  p.slopes = ctx->slopes_frame; p.lds = ctx->lds;
  return AOM_OK;
}

extern "C" int aom_comp_wfs_image(aom_ctx* ctx, int flags, float noise, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  if (noise >= 0.f && !ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must seed the noise streams first");
  WfsParams p;
  int rc = fill_wfs_params(ctx, p, flags, noise);
  if (rc) return rc;
  if (flags & 4) {
    if (!ctx->bincube) CU(dalloc(&ctx->bincube, (size_t)c.n_env * c.nvalid * 256));
    p.bincube = ctx->bincube;
  }
  // does any environment draw noise in this frame?  (host copies: no device read)
  bool noisy = p.noise >= 0.f && !p.noise_env;
  for (int e = 0; p.noise_env && e < c.n_env && !noisy; ++e) noisy = ctx->cond[AOM_COND_NOISE][0].host[e] >= 0.f;
  const bool timed = ctx->opt[AOM_OPT_TIME_WFS] && ctx->wev_n < AOM_WFS_TIMERS;
  if (timed)
    for (int j = 0; j < 2; ++j)
      if (!ctx->wev[j][ctx->wev_n]) CU(cudaEventCreate(&ctx->wev[j][ctx->wev_n]));
  rc = wfs_frame_launch(ctx->wfs, p, ctx->opt[AOM_OPT_WFS_PATH], noisy, timed ? ctx->wev[0][ctx->wev_n] : nullptr, st, ctx->err);
  if (rc) return rc;
  KCHECK();
  if (timed) {
    CU(cudaEventRecord(ctx->wev[1][ctx->wev_n], st));
    ctx->wev_n++;
  }
  if (!(flags & 8)) ctx->frame++;        // bit3: an extra look at the same frame (ROKET's noise-free image): noise stream untouched
  ctx->cube_override = nullptr;
  return AOM_OK;
}

extern "C" int aom_wfs_time_ms(aom_ctx* ctx, float* mean_ms, int* count) {
  if (!ctx || !mean_ms || !count) return fail(ctx, AOM_ERR_INVALID, "null argument");
  double sum = 0.0;
  for (int i = 0; i < ctx->wev_n; ++i) {
    float ms = 0.f;
    CU(cudaEventSynchronize(ctx->wev[1][i]));
    CU(cudaEventElapsedTime(&ms, ctx->wev[0][i], ctx->wev[1][i]));
    sum += ms;
  }
  *count = ctx->wev_n;
  *mean_ms = ctx->wev_n ? (float)(sum / ctx->wev_n) : 0.f;
  ctx->wev_n = 0;
  return AOM_OK;
}

extern "C" const char* aom_wfs_kernel(aom_ctx* ctx) {
  if (!ctx) return "";
  return wfs_frame_kernel_name(ctx->wfs, ctx->opt[AOM_OPT_WFS_PATH], ctx->err);
}

extern "C" int aom_raytrace_wfs(aom_ctx* ctx, int flags, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  WfsParams p;
  int rc = fill_wfs_params(ctx, p, flags, -1.f);
  if (rc) return rc;
  if (flags & AOM_TAR_GEO) {                       // through the geometric controller's mirrors instead of the main ones
    rc = geo_prepare(ctx);
    if (rc) return rc;
    p.volts = ctx->geo_volts;
  }
  if (!ctx->phase) CU(dalloc(&ctx->phase, (size_t)c.n_env * c.n * c.n));
  dim3 blk(32, 8), grid((c.n + 31) / 32, (c.n + 7) / 8, c.n_env);
  with<false, true>(p.wind != nullptr, [&](auto PE) { wfs_phase_kernel<PE><<<grid, blk, 0, st>>>(p, ctx->phase); });
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_do_centroids_geom(aom_ctx* ctx, int flags, float alpha, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  if (c.pdiam != 16) return fail(ctx, AOM_ERR_UNSUPPORTED, "geometric slopes need 16-pixel subapertures");
  int rc = aom_raytrace_wfs(ctx, flags, stream);
  if (rc) return rc;
  WfsParams p;
  rc = fill_wfs_params(ctx, p, flags, -1.f);
  if (rc) return rc;
  slopes_geom_kernel<<<dim3(c.nvalid, c.n_env), 256, 0, (cudaStream_t)stream>>>(p, ctx->phase, ctx->slopes, ctx->lds, alpha);
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_comp_strehl(aom_ctx* ctx, int flags, float lambda_um, int accumulate, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  if (!(lambda_um > 0.f)) return fail(ctx, AOM_ERR_INVALID, "target wavelength must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  WfsParams p;
  int rc = fill_wfs_params(ctx, p, flags, -1.f);
  if (rc) return rc;
  const bool geo = (flags & AOM_TAR_GEO) != 0;
  if (geo) {
    rc = geo_prepare(ctx);
    if (rc) return rc;
    p.volts = ctx->geo_volts;
  }
  int& n_le = geo ? ctx->geo_tar_n : ctx->tar_n;
  double* mom = ctx->tar_mom + (geo ? (size_t)c.n_env * PSW_MOM2 : 0);
  // AOM_TAR_PEAK: brightest pixel of the PSF core with a three-point fit (comp_strehl(do_fit=True)) instead of the
  // on-axis pixel; the pending sums remember which of the two a trace produced
  int& peak = geo ? ctx->geo_tar_peak : ctx->tar_peak;
  if (!(flags & AOM_TAR_PUBLISH)) {
    peak = (flags & AOM_TAR_PEAK) != 0 || ctx->opt[AOM_OPT_STREHL_PEAK] != 0;
    const int nfft = ctx->opt[AOM_OPT_PSF_NFFT];
    if (peak && nfft < c.n) return fail(ctx, AOM_ERR_STATE, "AOM_OPT_PSF_NFFT (focal-plane grid of the target, >= pupil size) is not set");
    CU(cudaMemsetAsync(mom, 0, (size_t)c.n_env * PSW_MOM2 * sizeof(double), st));
    rc = sweep_prepare(ctx, st);
    if (rc) return rc;
    const float k2t = (float)(2.0 * M_PI / (double)lambda_um);
    if (ctx->sweep_state == 1 && ctx->opt[AOM_OPT_PUPIL_PATH] == AOM_PUPIL_SWEEP) {
      rc = peak ? sweep_launch<2>(ctx, p, nullptr, mom, st, k2t, 1.f / (float)nfft) : sweep_launch<1>(ctx, p, nullptr, mom, st, k2t);
      if (rc) return rc;
    } else {
      dim3 blk(32, 8), grid((c.n + 31) / 32, (c.n + 7) / 8, c.n_env);
      with<false, true>(p.wind != nullptr, [&](auto PE) {
        target_moments_kernel<PE><<<grid, blk, 0, st>>>(p, mom, k2t, peak ? PSW_MOM2 : 5, peak ? 1.f / (float)nfft : 0.f);
      });
      KCHECK();
    }
    if (flags & AOM_TAR_TRACE) return AOM_OK;        // sums pending until AOM_TAR_PUBLISH
  }
  if (accumulate) n_le += 1;
  float* out = geo ? ctx->strehl_geo : ctx->strehl;
  float* acc = geo ? ctx->geo_acc : ctx->tar_acc;
  // staggered environments: their own long-exposure counts; one whose first step is pending is skipped
  int* le_n = ctx->staggered ? ctx->le_n + (geo ? c.n_env : 0) : nullptr;
  if (peak) target_strehl_core_kernel<<<(c.n_env + 127) / 128, 128, 0, st>>>(mom, out, acc, c.n_env, accumulate ? n_le : 0, le_n, ctx->first);
  else target_strehl_kernel<<<(c.n_env + 127) / 128, 128, 0, st>>>(mom, 5, out, acc, c.n_env, accumulate ? n_le : 0, le_n, ctx->first);
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_do_control_geo(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  NEED(AOM_T_GEO_PROJ, 0); NEED(AOM_T_GEO_SIFN, 0);
  int rc = geo_prepare(ctx);
  if (rc) return rc;
  WfsParams p;
  rc = fill_wfs_params(ctx, p, 1 | 2, -1.f);      // the mirrors' tables are needed, their voltages are not read
  if (rc) return rc;
  CU(cudaMemsetAsync(ctx->geo_mom, 0, (size_t)c.n_env * 4 * sizeof(double), st));
  rc = sweep_prepare(ctx, st);
  if (rc) return rc;
  int nb = 0;
  if (ctx->sweep_state == 1 && ctx->opt[AOM_OPT_PUPIL_PATH] == AOM_PUPIL_SWEEP) {
    rc = sweep_launch<0>(ctx, p, ctx->geo_T, ctx->geo_mom, st);
    if (rc) return rc;
    nb = ctx->sweep_nb;
  } else {
    const size_t smem = (size_t)GEO_ROW_WARPS * (c.n + (c.n >> 4) + 2) * sizeof(float);
    dim3 grid((c.n + GEO_ROW_WARPS - 1) / GEO_ROW_WARPS, c.n_env);
    with<false, true>(p.wind != nullptr, [&](auto PE) {
      geo_rows_kernel<PE><<<grid, GEO_ROW_WARPS * 32, smem, st>>>(p, ctx->geo_T, ctx->geo_gp, ctx->geo_mom);
    });
    KCHECK();
  }
  geo_cols_kernel<<<c.n_env, 256, 0, st>>>(p, ctx->geo_T, ctx->geo_gp, nb, ctx->geo_mom,
                                           (const float*)ctx->tab[AOM_T_GEO_SIFN][0], ctx->geo_b, ctx->lda);
  KCHECK();
  // exact float32 FFMA accumulation: the tip-tilt entries of b are 100x the piezo ones and the product cancels to
  // ~1e-3 of its largest terms; the tensor core's truncated accumulator left 3 % errors in the commands (measured,
  // profiles/dev/geo_probe.py).  The reference inverts and multiplies in double (sutra_controller_geo).
  GemmParams g;
  memset(&g, 0, sizeof(g));
  g.A = ctx->geo_b; g.lda = ctx->lda; g.B = (const float*)ctx->tab[AOM_T_GEO_PROJ][0]; g.ldb = ctx->lda;
  g.C = ctx->geo_com; g.ldc = ctx->lda; g.M = c.n_env; g.N = c.nactu; g.K = c.nactu;
  rc = gemm_launch(g, 0, 1, true, ctx->opt[AOM_OPT_GEMM_PATH], ctx->num_sms, ctx->d_err, st, ctx->err);
  if (rc) return rc;
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_apply_control_geo(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc = geo_prepare(ctx);
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->geo_volts, ctx->geo_com, (size_t)ctx->cfg.n_env * ctx->lda * sizeof(float),
                     cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return AOM_OK;
}

extern "C" int aom_reset_strehl(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  ctx->tar_n = 0;
  if (ctx->le_n) CU(cudaMemsetAsync(ctx->le_n, 0, (size_t)ctx->cfg.n_env * sizeof(int), (cudaStream_t)stream));
  CU(cudaMemsetAsync(ctx->tar_acc, 0, (size_t)ctx->cfg.n_env * TAR_ACC * sizeof(float), (cudaStream_t)stream));
  CU(cudaMemsetAsync(ctx->strehl, 0, (size_t)ctx->cfg.n_env * 4 * sizeof(float), (cudaStream_t)stream));
  if (ctx->geo_com) {
    ctx->geo_tar_n = 0;
    if (ctx->le_n) CU(cudaMemsetAsync(ctx->le_n + ctx->cfg.n_env, 0, (size_t)ctx->cfg.n_env * sizeof(int), (cudaStream_t)stream));
    CU(cudaMemsetAsync(ctx->geo_acc, 0, (size_t)ctx->cfg.n_env * TAR_ACC * sizeof(float), (cudaStream_t)stream));
    CU(cudaMemsetAsync(ctx->strehl_geo, 0, (size_t)ctx->cfg.n_env * 4 * sizeof(float), (cudaStream_t)stream));
  }
  return AOM_OK;
}

extern "C" int aom_set_bincube(aom_ctx* ctx, const float* dcube, void* stream) {
  if (!ctx || !dcube) return fail(ctx, AOM_ERR_INVALID, "null argument");
  (void)stream;
  ctx->cube_override = dcube;
  return AOM_OK;
}

extern "C" int aom_denoise(aom_ctx* ctx, const float* din, float* dout, long long n_spots, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  NEED(AOM_T_DENOISER, 0);
  const aom_config& c = ctx->cfg;
  if (!din) {
    if (!ctx->bincube) return fail(ctx, AOM_ERR_STATE, "no detector cube: run aom_comp_wfs_image with the keep-image flag first");
    din = ctx->bincube;
    n_spots = (long long)c.n_env * c.nvalid;
  }
  if (n_spots < 0) return fail(ctx, AOM_ERR_INVALID, "negative spot count");
  const bool in_place = dout == nullptr;
  if (in_place) {
    if (din != ctx->bincube) return fail(ctx, AOM_ERR_INVALID, "in-place denoising needs the context's detector cube as input");
    dout = ctx->bincube;
  }
  if (n_spots > 0 && ctx->opt[AOM_OPT_DENOISE_PATH] == AOM_DENOISE_TCGEN05 && ctx->tab[AOM_T_DENOISER_TC][0]) {
    DnTcParams P;
    P.in = din; P.out = dout; P.n_spots = n_spots;
    P.wblob = (const uint8_t*)ctx->tab[AOM_T_DENOISER_TC][0] + (size_t)DT_NPARAM * 4;
    P.err = ctx->d_err;
    P.dbg = getenv("AOM_DN_TIMING") ? ctx->dn_dbg : nullptr;
    memcpy(P.prm, ctx->dn_prm, sizeof(P.prm));
    CU(denoise_tc_launch(P, ctx->num_sms, (cudaStream_t)stream));
    ctx->launches += 1;
    if (P.dbg) {   // development: per-phase clock totals of CTA 0
      long long h[32];
      CU(cudaStreamSynchronize((cudaStream_t)stream));
      CU(cudaMemcpy(h, ctx->dn_dbg, sizeof(h), cudaMemcpyDeviceToHost));
      const char* nm[9] = {"load+e1", "e2 mma", "e2 epi", "e3 mma", "e3 epi", "d1 mma", "d1 epi", "d2 mma", "d2 epi+d3+store"};
      const double passes = (double)((n_spots + DT_G - 1) / DT_G + ctx->num_sms - 1) / ctx->num_sms;
      for (int i = 0; i < 9; ++i) fprintf(stderr, "denoise_tc %-16s %9.0f cycles per pass\n", nm[i], (double)h[i] / passes);
      const char* cn[15] = {"e2 wait w", "e2 issue", "e2 complete", "e3 wait w hi", "e3 issue hi", "e3 wait w lo", "e3 issue lo", "e3 complete",
                            "d1 wait w (4x)", "d1 issue (4x)", "d1 wait class + reload (2x)", "d1 complete", "d2 wait w", "d2 issue", "d2 complete"};
      for (int i = 0; i < 15; ++i) fprintf(stderr, "denoise_tc issuing lane: %-28s %9.0f cycles per pass\n", cn[i], (double)h[16 + i] / passes);
    }
  } else if (n_spots > 0) {
    CU(cudaFuncSetAttribute(denoise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DN_SMEM_BYTES));
    const long long batches = (n_spots + DN_G - 1) / DN_G;
    const int grid = (int)(batches < ctx->num_sms ? batches : ctx->num_sms);
    denoise_kernel<<<grid, DN_THREADS, DN_SMEM_BYTES, (cudaStream_t)stream>>>(din, dout, n_spots,
                                                                              (const float*)ctx->tab[AOM_T_DENOISER][0]);
    KCHECK();
  }
  if (in_place) ctx->cube_override = ctx->bincube;
  return AOM_OK;
}

extern "C" int aom_do_centroids(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  if (ctx->cube_override) {
    long long total = (long long)c.n_env * c.nvalid;
    long long threads = total * 32;
    cog_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(ctx->cube_override, ctx->slopes, ctx->lds, c.nvalid,
                                                                  total, c.cog_offset, c.pixsize);
    KCHECK();
  } else {
    CU(cudaMemcpyAsync(ctx->slopes, ctx->slopes_frame, (size_t)c.n_env * ctx->lds * 4, cudaMemcpyDeviceToDevice, st));
  }
  return AOM_OK;
}

extern "C" int aom_do_control(aom_ctx* ctx, void* stream) {
  return ctx ? rtc_do_control(ctx->rtc, ctx->slopes, (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

extern "C" int aom_set_command(aom_ctx* ctx, const float* dcom, int ld, void* stream) {
  if (!ctx || !dcom) return fail(ctx, AOM_ERR_INVALID, "null argument");
  return rtc_set_rows(ctx->rtc, AOM_B_COM, dcom, ld, (cudaStream_t)stream, ctx->err);
}

extern "C" int aom_set_dm_volts(aom_ctx* ctx, const float* dvolts, int ld, void* stream) {
  if (!ctx || !dvolts) return fail(ctx, AOM_ERR_INVALID, "null argument");
  return rtc_set_rows(ctx->rtc, AOM_B_VOLTS, dvolts, ld, (cudaStream_t)stream, ctx->err);
}

extern "C" int aom_apply_control(aom_ctx* ctx, int comp_voltage, void* stream) {
  return ctx ? rtc_apply_control(ctx->rtc, comp_voltage, (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

extern "C" int aom_set_option(aom_ctx* ctx, int option, int value) {
  if (!ctx) return AOM_ERR_INVALID;
  if (option < 0 || option >= AOM_OPT_COUNT) return fail(ctx, AOM_ERR_INVALID, "unknown option %d", option);
  if (option == AOM_OPT_WFS_PATH && (value < 0 || value > AOM_WFS_UMMA_WS))
    return fail(ctx, AOM_ERR_INVALID, "AOM_OPT_WFS_PATH: value %d out of range", value);
  if (option == AOM_OPT_TIME_WFS) ctx->wev_n = 0;
  if (option == AOM_OPT_GEMM_PATH && (value < 0 || value > AOM_GEMM_TF32))
    return fail(ctx, AOM_ERR_INVALID, "AOM_OPT_GEMM_PATH: value %d out of range", value);
  ctx->opt[option] = value;
  return AOM_OK;
}

extern "C" int aom_check_device(aom_ctx* ctx) {
  if (!ctx) return AOM_ERR_INVALID;
  int h = 0;
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(&h, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost));
  if (h) {
    CU(cudaMemset(ctx->d_err, 0, sizeof(int)));
    return fail(ctx, AOM_ERR_CUDA, "device error word %d: a bounded mbarrier wait expired in gemm_tc_kernel", h);
  }
  return AOM_OK;
}

extern "C" int aom_set_gain(aom_ctx* ctx, float gain) {
  const CondSet s = {AOM_COND_GAIN, 0, false, &gain};
  return set_conditions(ctx, 1, &s);
}

extern "C" int aom_set_gain_env(aom_ctx* ctx, const float* gain_host) {
  const CondSet s = {AOM_COND_GAIN, 0, true, gain_host};
  return set_conditions(ctx, 1, &s);
}

extern "C" int aom_set_delay(aom_ctx* ctx, float delay) {
  const CondSet s = {AOM_COND_DELAY, 0, false, &delay};
  return set_conditions(ctx, 1, &s);
}

extern "C" int aom_set_delay_env(aom_ctx* ctx, const float* delay_host) {
  const CondSet s = {AOM_COND_DELAY, 0, true, delay_host};
  return set_conditions(ctx, 1, &s);
}

extern "C" int aom_set_wfs_noise(aom_ctx* ctx, float noise, float nphotons) {
  const CondSet s[2] = {{AOM_COND_NOISE, 0, false, &noise}, {AOM_COND_NPHOTONS, 0, false, &nphotons}};
  return set_conditions(ctx, 2, s);
}

extern "C" int aom_set_wfs_noise_env(aom_ctx* ctx, const float* noise_host, const float* nphotons_host) {
  const CondSet s[2] = {{AOM_COND_NOISE, 0, true, noise_host}, {AOM_COND_NPHOTONS, 0, true, nphotons_host}};
  return set_conditions(ctx, 2, s);
}

extern "C" int aom_set_loop(aom_ctx* ctx, int closed) {
  if (!ctx) return AOM_ERR_INVALID;
  rtc_set_loop(ctx->rtc, closed);
  return AOM_OK;
}

extern "C" int aom_set_layer(aom_ctx* ctx, int layer, float deltax, float deltay, float amp) {
  const CondSet s[3] = {{AOM_COND_WIND_X, layer, false, &deltax}, {AOM_COND_WIND_Y, layer, false, &deltay},
                        {AOM_COND_AMP, layer, false, &amp}};
  return set_conditions(ctx, 3, s);
}

extern "C" int aom_set_layer_amp(aom_ctx* ctx, int layer, const float* amp_host) {
  const CondSet s = {AOM_COND_AMP, layer, true, amp_host};
  return set_conditions(ctx, 1, &s);
}

extern "C" int aom_reset_dm(aom_ctx* ctx, void* stream) {
  return ctx ? rtc_reset_dm(ctx->rtc, (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

// The counters of this context that the controller's half-steps read
static RtcCounters counters(const aom_ctx* ctx) {
  return RtcCounters{ctx->step, ctx->staggered ? ctx->step_env : nullptr, ctx->first, ctx->first_any};
}

extern "C" int aom_rl_control(aom_ctx* ctx, const float* daction, void* stream) {
  return ctx ? rtc_rl_control(ctx->rtc, daction, counters(ctx), (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

extern "C" int aom_state_begin(aom_ctx* ctx, void* stream) {
  return ctx ? rtc_state_begin(ctx->rtc, (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

// The linear half-step of environments restarted by aom_reset_envs is done: their next rl half-step is an ordinary one.
static int end_first_steps(aom_ctx* ctx, cudaStream_t st) {
  if (!ctx->first_any) return AOM_OK;
  CU(cudaMemsetAsync(ctx->first, 0, (size_t)ctx->cfg.n_env * sizeof(int), st));
  ctx->first_any = false;
  return AOM_OK;
}

extern "C" int aom_state_end(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc = rtc_state_end(ctx->rtc, (cudaStream_t)stream, ctx->err);
  return rc ? rc : end_first_steps(ctx, (cudaStream_t)stream);
}

extern "C" int aom_reward(aom_ctx* ctx, float factor, void* stream) {
  return ctx ? rtc_reward(ctx->rtc, factor, (cudaStream_t)stream, ctx->err) : AOM_ERR_INVALID;
}

extern "C" int aom_actor_forward(aom_ctx* ctx, int eval_mode, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc = rtc_actor_forward(ctx->rtc, eval_mode, counters(ctx), (cudaStream_t)stream, ctx->err);
  if (rc) return rc;
  ctx->step++;      // one decision per call: the exploration-noise counter (oracle/rng.py TAG_ACTOR)
  return AOM_OK;
}

extern "C" int aom_step(aom_ctx* ctx, int mode, int eval_mode, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  int rc;
  cudaStream_t st = (cudaStream_t)stream;
  // The turbulence update (exact-fp32 extrusion GEMMs on the FP32 pipe) touches only the screens, the rl
  // half-step (tensor-core GEMMs of the actors and the modal projections) only the controller state: they run
  // side by side on two streams and join before the sensor frame.
  const bool atmos_done = (mode & AOM_STEP_ATMOS_DONE) != 0;
  mode &= ~AOM_STEP_ATMOS_DONE;
  // with the per-frame Strehl the target sweep reads the screens of the previous frame after apply_control, so the
  // turbulence update cannot run ahead of it: no fork, no caller-side update
  const int strehl = ctx->opt[AOM_OPT_STREHL];
  if (strehl && atmos_done)
    return fail(ctx, AOM_ERR_STATE, "AOM_OPT_STREHL needs the screens of the previous frame: do not combine with AOM_STEP_ATMOS_DONE");
  const bool fork = ctx->cfg.n_layers > 0 && ctx->seeded && !atmos_done && !strehl;
  if (fork) {
    CU(cudaEventRecord(ctx->ev_fork, st));
    CU(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0));
    rc = aom_move_atmos(ctx, ctx->side_stream); if (rc) return rc;
    CU(cudaEventRecord(ctx->ev_join, ctx->side_stream));
  }
  // rl half-step: TrainerRPC.env_step -> AoEnv.rl_step -> RlSupervisor.next_part_two (rlSupervisor.py:900-947)
  if (mode == 0) { rc = aom_actor_forward(ctx, eval_mode, stream); if (rc) return rc; }
  if (mode != 2) { rc = aom_rl_control(ctx, nullptr, stream); if (rc) return rc; }
  // next_part_two: target.comp_tar_image + comp_strehl (rlSupervisor.py:936-947).  The atmosphere is still the one of
  // the previous frame; the mirrors carry the voltages the target was traced with in next_part_one (option value 1:
  // before apply_control) or, with "pure delay 0", the new ones (value 2: re-traced after apply_control)
  const int nm = ctx->opt[AOM_OPT_STREHL_LAMBDA_NM] > 0 ? ctx->opt[AOM_OPT_STREHL_LAMBDA_NM] : 1650;
  if (strehl == 1) { rc = aom_comp_strehl(ctx, 3, (float)nm * 1e-3f, 1, stream); if (rc) return rc; }
  rc = aom_apply_control(ctx, 1, stream); if (rc) return rc;
  if (strehl >= 2) { rc = aom_comp_strehl(ctx, 3, (float)nm * 1e-3f, 1, stream); if (rc) return rc; }
  const RtcView v = rtc_view(ctx->rtc);
  if (v.reward) { rc = aom_reward(ctx, ctx->cfg.reward_factor, stream); if (rc) return rc; }
  // linear half-step: AoEnv.linear_step -> RlSupervisor.next_part_one (rlSupervisor.py:1015-1051)
  rc = aom_state_begin(ctx, stream); if (rc) return rc;
  if (fork) CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
  else if (!atmos_done) { rc = aom_move_atmos(ctx, stream); if (rc) return rc; }
  // second controller of the production parameter files (next_part_one loops over p_controllers,
  // rlSupervisor.py:1036-1046): it reads only the moved screens, so it runs beside the sensor frame
  const bool geo = ctx->opt[AOM_OPT_GEO] != 0;
  if (geo) {
    cudaStream_t gs = fork ? ctx->side_stream : st;
    rc = aom_do_control_geo(ctx, gs); if (rc) return rc;
    rc = aom_apply_control_geo(ctx, gs); if (rc) return rc;
    if (fork) CU(cudaEventRecord(ctx->ev_geo, gs));
  }
  const bool denoise = ctx->opt[AOM_OPT_DENOISE] != 0;
  const bool keep = denoise || ctx->opt[AOM_OPT_KEEP_IMAGE] != 0;
  // the common noise, or with per-environment noise in force any value >= 0: each environment's own
  const EnvCond& noise = ctx->cond[AOM_COND_NOISE][0];
  rc = aom_comp_wfs_image(ctx, keep ? 7 : 3, noise.dev ? 0.f : noise.common, stream); if (rc) return rc;
  if (denoise) { rc = aom_denoise(ctx, nullptr, nullptr, 0, stream); if (rc) return rc; }
  rc = aom_do_centroids(ctx, stream); if (rc) return rc;
  rc = aom_do_control(ctx, stream); if (rc) return rc;
  if (v.state) { rc = aom_state_end(ctx, stream); if (rc) return rc; }
  else { rc = end_first_steps(ctx, st); if (rc) return rc; }
  if (geo && fork) CU(cudaStreamWaitEvent(st, ctx->ev_geo, 0));
  return AOM_OK;
}

extern "C" int aom_pixel_noise(aom_ctx* ctx, const float* dlam, float* dout, int64_t n, float noise, int64_t seed,
                               uint32_t frame, uint32_t wfs, void* stream) {
  if (!ctx || !dlam || !dout) return fail(ctx, AOM_ERR_INVALID, "null argument");
  uint64_t s = (uint64_t)seed;
  pixel_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dlam, dout, n, noise, (uint32_t)(s & 0xffffffffu),
                                                                                   (uint32_t)(s >> 32), frame, wfs);
  KCHECK();
  return AOM_OK;
}
