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
#include "atmos_kernels.cuh"
#include "gemm_kernels.cuh"
#include "gemm_tc.cuh"
#include "rtc_kernels.cuh"
#include "wfs_kernels.cuh"
#include "wfs_mma.cuh"
#include "wfs_lattice_host.h"
#include "wfs_tma.cuh"
#include "wfs_umma_host.h"
#include "extrude_i8_host.h"
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
  // atmosphere
  float* screen[AOM_MAX_LAYERS];
  int* ox[AOM_MAX_LAYERS];
  int* oy[AOM_MAX_LAYERS];
  uint32_t* ext_count[AOM_MAX_LAYERS];
  float* amp_env[AOM_MAX_LAYERS];     // optional per-environment innovation amplitude (aom_set_layer_amp)
  double accx[AOM_MAX_LAYERS], accy[AOM_MAX_LAYERS];
  // per-environment winds (aom_set_layer_wind).  While wind_pe is set every layer keeps one accumulator per environment
  // on the device (wind_state_kernel) and in a host mirror that only sizes the extrusion passes; the extrusion and
  // sampling kernels run their per-environment instantiations.  Otherwise accx / accy above hold the state.
  float *wind_dx[AOM_MAX_LAYERS], *wind_dy[AOM_MAX_LAYERS];     // device [E] steps of layers with their own winds, else null
  float *wind_hdx[AOM_MAX_LAYERS], *wind_hdy[AOM_MAX_LAYERS];   // host copies
  bool wind_pe;
  double* wind_acc;            // device [L][2][E] accumulators (x, y)
  int* wind_steps;             // device [L][2][E] whole-pixel counts of the last frame (x, y)
  WindRec* wind_rec;           // device [L][E] offsets for the samplers
  double* wind_hacc;           // host mirror of wind_acc
  int wind_passes[AOM_MAX_LAYERS][2];   // extrusion passes of the last frame: max over the batch of |count| (x, y)
  int wind_box[AOM_MAX_LAYERS][4];      // min / max over the batch of ix, then of iy (pupil footprint check)
  uint32_t *k0, *k1;
  float *Z, *zref, *newcol;
  int ldz_max, ldn_max;
  // exact integer extrusion (extrude_i8.cuh): operator digit planes per layer, environment digit planes, row scales
  uint8_t* oz_ab[AOM_MAX_LAYERS];
  int* oz_ea[AOM_MAX_LAYERS];
  int oz_kb[AOM_MAX_LAYERS], oz_nt[AOM_MAX_LAYERS];
  uint8_t* oz_zs;
  int* oz_ev;
  size_t oz_zs_bytes;
  // the same integer contraction for the controller's operator products (cmat, v2m, m2v): operator digit planes per
  // table, scratch digit planes of the per-environment vectors (main stream; the extrusion has its own on the side stream)
  uint8_t* ozop[AOM_T_COUNT];
  int* ozop_ea[AOM_T_COUNT];
  int ozop_kb[AOM_T_COUNT], ozop_nt[AOM_T_COUNT];
  uint8_t* oz_xs;
  int* oz_xev;
  size_t oz_xs_bytes;
  // actor weights as pre-split TF32 hi / lo planes in the tile order of gemm_tc_kernel (W1, W2, WH), floats per agent
  float* actor_bt[3];
  size_t actor_bt_per[3];
  // sensor / rtc
  float *slopes_frame, *slopes, *err_v, *com, *com1, *volts, *com_before;
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
  int lds, lda, ldm;
  float gain;
  int closed;
  uint32_t frame;
  // sensor noise / photon count / integrator gain: common values (aom_set_wfs_noise, aom_set_gain) and optional
  // per-environment ones (aom_set_wfs_noise_env, aom_set_gain_env): device [E] arrays while in force, else null, with
  // host copies that route the frames without a device read
  float noise_c, nph_c;
  float *noise_env, *nph_env, *gain_env;
  float *noise_henv, *nph_henv, *gain_henv;
  int opt[AOM_OPT_COUNT];
  long long* dn_dbg;
  float dn_prm[DT_NPARAM];    // float parameters of the tensor-core denoiser (head of AOM_T_DENOISER_TC)
  int tar_peak, geo_tar_peak; // whether the pending target sums hold the PSF core (AOM_TAR_PEAK)
  int* d_err;                 // device error word raised by bounded waits (gemm_tc.cuh)
  // RL
  float *modes, *modes_before, *modes_res, *state, *hist, *reward, *action, *action_mean, *strehl;
  int ldst, ldact, hist_head;
  uint32_t step;
  float *aX, *aH1, *aH2, *aHO;
  int ld_ain, ld_ah, ld_aho;
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
  // staged Shack-Hartmann kernels: host copies of the tables their own tables derive from; fast_why says why the last
  // refused preparation refused
  void* htab[AOM_T_COUNT];
  size_t htab_bytes[AOM_T_COUNT];
  char fast_why[160];
  // TMA-staged kernel (wfs_tma.cuh): derived tables
  int fast_state;            // 0 = not prepared, 1 = eligible, -1 = not eligible
  WfsFast fast;
  void* fast_dev[6];
  CUtensorMap fast_maps[WFT_MAX_LAYERS];
  // tcgen05 kernels (wfs_umma.cuh, wfs_umma_ws.cuh): derived tables
  int umma_state;            // 0 = not prepared, 1 = eligible, -1 = not eligible
  WfsUmmaHost umma;
  void* umma_dev[6];
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

template <typename T>
static cudaError_t dalloc(T** p, size_t count) {
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e == cudaSuccess) e = cudaMemset(*p, 0, count * sizeof(T));
  // the fill runs on the legacy stream, the buffer may be used next on a non-blocking one: finish it here
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  return e;
}

// Kernels launched with more dynamic shared memory than the default: f(kernel, bytes, its template arguments) for every
// instantiation.  aom_create sets the attribute of each and the launch sites launch from the same lists.
template <class F>
static void gemm_tc_each(F&& f) {     // tcgen05 GEMM: epilogue, column tile
  each<0, 1, 2>([&](auto EPI) {
    each<GTC_BN, GTC_BN_WIDE>([&](auto BN) { f(gemm_tc_kernel<EPI, BN>, (size_t)GTC_SMEM_BYTES_T(BN), EPI, BN); });
  });
}

template <class F>
static void wfs_simt_each(F&& f) {    // SIMT sensor frame: Nfft / 16, per-environment winds, per-environment sensor values
  each<4, 8>([&](auto R) {
    each<false, true>([&](auto PE) { each<false, true>([&](auto NE) { f(wfs_frame_kernel<R, PE, NE>, wfs_smem_bytes<R>(), R, PE, NE); }); });
  });
}

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
  if (cfg->delay != 0 && cfg->delay != 1) return fail(nullptr, AOM_ERR_UNSUPPORTED, "controller delay must be 0 or 1 frame");

  // the context embeds CUtensorMap objects (64-byte aligned)
  ctx = (aom_ctx*)aligned_alloc(64, (sizeof(aom_ctx) + 63) / 64 * 64);
  if (!ctx) return fail(nullptr, AOM_ERR_INVALID, "out of host memory");
  memset(ctx, 0, sizeof(aom_ctx));
  ctx->cfg = *cfg;
  ctx->gain = cfg->gain;
  ctx->noise_c = cfg->noise;
  ctx->nph_c = cfg->nphotons;
  ctx->closed = 1;
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
  ctx->ldm = AOM_LD(cfg->nmodes > 0 ? cfg->nmodes : 1);
  for (int l = 0; l < cfg->n_layers; ++l) {
    size_t N = cfg->screen_dim[l];
    CU(dalloc(&ctx->screen[l], E * N * N));
    CU(dalloc(&ctx->ox[l], E));
    CU(dalloc(&ctx->oy[l], E));
    CU(dalloc(&ctx->ext_count[l], E));
    int ldz = AOM_LD(cfg->stencil_size[l] + (int)N);
    if (ldz > ctx->ldz_max) ctx->ldz_max = ldz;
    if (AOM_LD((int)N) > ctx->ldn_max) ctx->ldn_max = AOM_LD((int)N);
  }
  CU(dalloc(&ctx->k0, E));
  CU(dalloc(&ctx->k1, E));
  if (cfg->n_layers > 0) {
    CU(dalloc(&ctx->Z, E * ctx->ldz_max));
    CU(dalloc(&ctx->zref, E));
    CU(dalloc(&ctx->newcol, E * ctx->ldn_max));
  }
  CU(dalloc(&ctx->slopes_frame, E * ctx->lds));
  CU(dalloc(&ctx->slopes, E * ctx->lds));
  CU(dalloc(&ctx->err_v, E * ctx->lda));
  CU(dalloc(&ctx->com, E * ctx->lda));
  CU(dalloc(&ctx->com1, E * ctx->lda));
  CU(dalloc(&ctx->volts, E * ctx->lda));
  CU(dalloc(&ctx->com_before, E * ctx->lda));
  CU(dalloc(&ctx->strehl, E * 4));
  CU(dalloc(&ctx->tar_mom, E * 2 * PSW_MOM2));     // main target, then the geometric controller's
  CU(dalloc(&ctx->tar_acc, E * TAR_ACC));
  CU(cudaMalloc((void**)&ctx->dn_dbg, 32 * sizeof(long long)));
  if (cfg->nmodes > 0) {
    CU(dalloc(&ctx->modes, E * ctx->ldm));
    CU(dalloc(&ctx->modes_before, E * ctx->ldm));
    CU(dalloc(&ctx->modes_res, E * ctx->ldm));
  }
  if (cfg->state_dim > 0) {
    ctx->ldst = AOM_LD(cfg->state_dim);
    CU(dalloc(&ctx->state, E * ctx->ldst));
    if (cfg->n_hist > 0) CU(dalloc(&ctx->hist, (size_t)cfg->n_hist * E * cfg->state_modes));
  }
  if (cfg->action_dim > 0) {
    ctx->ldact = AOM_LD(cfg->action_dim);
    CU(dalloc(&ctx->action, E * ctx->ldact));
    CU(dalloc(&ctx->action_mean, E * ctx->ldact));
  }
  if (cfg->n_agents > 0) {
    CU(dalloc(&ctx->reward, E * cfg->n_agents));
    ctx->ld_ain = AOM_LD(cfg->actor_in);
    ctx->ld_ah = AOM_LD(cfg->actor_hidden);
    ctx->ld_aho = AOM_LD(2 * cfg->actor_out);
    size_t A = cfg->n_agents;
    CU(dalloc(&ctx->aX, A * E * ctx->ld_ain));
    CU(dalloc(&ctx->aH1, A * E * ctx->ld_ah));
    CU(dalloc(&ctx->aH2, A * E * ctx->ld_ah));
    CU(dalloc(&ctx->aHO, A * E * ctx->ld_aho));
  }
  CU(dalloc(&ctx->d_err, 1));
  CU(cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  cudaError_t ae = cudaSuccess;
  auto smem_attr = [&](auto kernel, size_t smem, auto...) {
    if (ae == cudaSuccess) ae = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  };
  gemm_tc_each(smem_attr);
  wfs_simt_each(smem_attr);
  if (ae != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "cudaFuncSetAttribute(dynamic shared memory) failed: %s", cudaGetErrorString(ae));
  return AOM_OK;
}

extern "C" void aom_destroy(aom_ctx* ctx) {
  if (!ctx) return;
  for (int t = 0; t < AOM_T_COUNT; ++t)
    for (int l = 0; l < AOM_MAX_LAYERS; ++l) cudaFree(ctx->tab[t][l]);
  for (int l = 0; l < AOM_MAX_LAYERS; ++l) {
    cudaFree(ctx->screen[l]); cudaFree(ctx->ox[l]); cudaFree(ctx->oy[l]); cudaFree(ctx->ext_count[l]);
    cudaFree(ctx->amp_env[l]);
    cudaFree(ctx->wind_dx[l]); cudaFree(ctx->wind_dy[l]); free(ctx->wind_hdx[l]); free(ctx->wind_hdy[l]);
  }
  cudaFree(ctx->wind_acc); cudaFree(ctx->wind_steps); cudaFree(ctx->wind_rec); free(ctx->wind_hacc);
  cudaFree(ctx->noise_env); cudaFree(ctx->nph_env); cudaFree(ctx->gain_env);
  free(ctx->noise_henv); free(ctx->nph_henv); free(ctx->gain_henv);
  void* bufs[] = {ctx->k0, ctx->k1, ctx->Z, ctx->zref, ctx->newcol, ctx->slopes_frame, ctx->slopes, ctx->err_v,
                  ctx->com, ctx->com1, ctx->volts, ctx->com_before, ctx->bincube, ctx->phase, ctx->modes,
                  ctx->modes_before, ctx->modes_res, ctx->state, ctx->hist, ctx->reward, ctx->action,
                  ctx->action_mean, ctx->strehl, ctx->tar_mom, ctx->tar_acc, ctx->aX, ctx->aH1, ctx->aH2, ctx->aHO, ctx->d_err,
                  ctx->geo_com, ctx->geo_volts, ctx->geo_b, ctx->geo_T, ctx->strehl_geo, ctx->geo_acc, ctx->geo_mom,
                  ctx->sweep_mask, ctx->sweep_ttp, ctx->rs_envs, ctx->rs_seeds, ctx->frame0, ctx->step_env,
                  ctx->le_n, ctx->first};
  for (void* b : bufs) cudaFree(b);
  for (int l = 0; l < AOM_MAX_LAYERS; ++l) { cudaFree(ctx->oz_ab[l]); cudaFree(ctx->oz_ea[l]); }
  for (int t = 0; t < AOM_T_COUNT; ++t) { cudaFree(ctx->ozop[t]); cudaFree(ctx->ozop_ea[t]); }
  cudaFree(ctx->oz_zs); cudaFree(ctx->oz_ev); cudaFree(ctx->oz_xs); cudaFree(ctx->oz_xev);
  for (int i = 0; i < 3; ++i) cudaFree(ctx->actor_bt[i]);

  for (void* b : ctx->fast_dev) cudaFree(b);
  for (void* b : ctx->umma_dev) cudaFree(b);
  for (int i = 0; i < AOM_WFS_TIMERS; ++i)
    for (int j = 0; j < 2; ++j)
      if (ctx->wev[j][i]) cudaEventDestroy(ctx->wev[j][i]);
  if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_geo) cudaEventDestroy(ctx->ev_geo);
  for (int t = 0; t < AOM_T_COUNT; ++t) free(ctx->htab[t]);
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

// digit planes of an operator [rows][ld] (K valid columns) for the integer contraction (extrude_i8.cuh)
static int oz_upload_operator(aom_ctx* ctx, const float* host, int rows, int ld, int K, uint8_t** planes_d, int** ea_d,
                              int* kb_out, int* nt_out) {
  if (!oz_operator_finite(host, rows, ld, K)) return fail(ctx, AOM_ERR_INVALID, "operator table holds a NaN or an infinity");
  const int KB = (K + OZ_BK - 1) / OZ_BK, NT = (rows + OZ_BN - 1) / OZ_BN;
  const size_t bytes = (size_t)NT * KB * OZ_SLICES_B * OZ_B_TILE;
  uint8_t* planes = (uint8_t*)calloc(bytes, 1);
  int* ea = (int*)calloc((size_t)NT * OZ_BN, sizeof(int));
  if (!planes || !ea) { free(planes); free(ea); return fail(ctx, AOM_ERR_INVALID, "out of host memory"); }
  oz_slice_operator(host, rows, ld, K, KB, NT, planes, ea);
  cudaFree(*planes_d); cudaFree(*ea_d);
  *planes_d = nullptr; *ea_d = nullptr;
  cudaError_t e = cudaMalloc((void**)planes_d, bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**)ea_d, (size_t)NT * OZ_BN * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(*planes_d, planes, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(*ea_d, ea, (size_t)NT * OZ_BN * sizeof(int), cudaMemcpyHostToDevice);
  free(planes); free(ea);
  if (e != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "operator digit planes: %s", cudaGetErrorString(e));
  *kb_out = KB; *nt_out = NT;
  return AOM_OK;
}

extern "C" int aom_set_table(aom_ctx* ctx, int table, int index, const void* host, size_t nbytes) {
  if (!ctx || !host) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (table < 0 || table >= AOM_T_COUNT || index < 0 || index >= AOM_MAX_LAYERS)
    return fail(ctx, AOM_ERR_INVALID, "table id %d / index %d out of range", table, index);
  size_t want = table_expected_bytes(ctx, table, index);
  if (want != nbytes)
    return fail(ctx, AOM_ERR_INVALID, "Dimension mismatch: table %d[%d] expects %zu bytes, got %zu", table, index, want, nbytes);
  // operators of the integer contraction first: a non-finite one is refused before anything changes
  if (table == AOM_T_AB) {
    // digit planes of [A | B] for the exact integer extrusion
    const aom_config& c = ctx->cfg;
    const int N = c.screen_dim[index], K = c.stencil_size[index] + N;
    int rc = oz_upload_operator(ctx, (const float*)host, N, AOM_LD(K), K, &ctx->oz_ab[index], &ctx->oz_ea[index],
                                &ctx->oz_kb[index], &ctx->oz_nt[index]);
    if (rc) return rc;
  }
  if (table == AOM_T_CMAT || table == AOM_T_V2M || table == AOM_T_M2V) {
    // digit planes of the controller operators for the exact integer products
    const aom_config& c = ctx->cfg;
    const int rows = table == AOM_T_V2M ? c.nmodes : c.nactu;
    const int K = table == AOM_T_CMAT ? c.nslopes : table == AOM_T_V2M ? c.nactu : c.nmodes;
    int rc = oz_upload_operator(ctx, (const float*)host, rows, AOM_LD(K), K, &ctx->ozop[table], &ctx->ozop_ea[table],
                                &ctx->ozop_kb[table], &ctx->ozop_nt[table]);
    if (rc) return rc;
  }
  if (ctx->tab[table][index]) { cudaFree(ctx->tab[table][index]); ctx->tab[table][index] = nullptr; }
  CU(cudaMalloc(&ctx->tab[table][index], nbytes ? nbytes : 4));
  CU(cudaMemcpy(ctx->tab[table][index], host, nbytes, cudaMemcpyHostToDevice));
  ctx->tab_bytes[table][index] = nbytes;
  if (table == AOM_T_MPUPIL || table == AOM_T_SUB_X0 || table == AOM_T_SUB_Y0 || table == AOM_T_STAMP1D ||
      table == AOM_T_ACT_MAP || table == AOM_T_HALFXY || table == AOM_T_TT_PLANES) {
    free(ctx->htab[table]);
    ctx->htab[table] = malloc(nbytes ? nbytes : 4);
    if (!ctx->htab[table]) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    memcpy(ctx->htab[table], host, nbytes);
    ctx->htab_bytes[table] = nbytes;
    ctx->fast_state = 0;     // derived tables of the staged sensor kernels are rebuilt on the next frame
    ctx->umma_state = 0;
  }
  if (table == AOM_T_MPUPIL || table == AOM_T_TT_PLANES) ctx->sweep_state = 0;
  if (table == AOM_T_DENOISER_TC) memcpy(ctx->dn_prm, host, (size_t)DT_NPARAM * 4);   // float parameters travel as kernel arguments
  if (table == AOM_T_ACTOR_W1 || table == AOM_T_ACTOR_W2 || table == AOM_T_ACTOR_WH) {
    // the same weights pre-split into TF32 hi / lo planes in the tile order of gemm_tc_kernel: the actor GEMMs then take
    // their B operand by one bulk copy per stage instead of global loads + split + st.shared in the loader warps
    const aom_config& c = ctx->cfg;
    const int i = table == AOM_T_ACTOR_W1 ? 0 : table == AOM_T_ACTOR_W2 ? 1 : 2;
    const int K = i == 0 ? c.actor_in : c.actor_hidden, ldb = AOM_LD(K);
    const int rows = i == 2 ? 2 * c.actor_out : c.actor_hidden;
    const int ldc = AOM_LD(rows);                                   // the output's leading dimension fixes the n tiles
    const size_t per = gtc_pretile_floats(ldc, AOM_LD(K));
    float* h = (float*)calloc(per * (size_t)c.n_agents, sizeof(float));
    if (!h) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    gtc_pretile_host((const float*)host, c.n_agents, (long long)rows * ldb, ldb, rows, ldc, AOM_LD(K), h);
    cudaFree(ctx->actor_bt[i]); ctx->actor_bt[i] = nullptr;
    cudaError_t e = cudaMalloc((void**)&ctx->actor_bt[i], per * c.n_agents * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(ctx->actor_bt[i], h, per * c.n_agents * sizeof(float), cudaMemcpyHostToDevice);
    free(h);
    if (e != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "pre-tiled actor weights: %s", cudaGetErrorString(e));
    ctx->actor_bt_per[i] = per;
  }
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
  void* p = nullptr;
  size_t n = 0;
  switch (buffer) {
    case AOM_B_SCREEN:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = ctx->screen[index]; n = E * c.screen_dim[index] * c.screen_dim[index]; break;
    case AOM_B_RING_OX:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = ctx->ox[index]; n = E; break;
    case AOM_B_RING_OY:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = ctx->oy[index]; n = E; break;
    case AOM_B_EXT_COUNT:
      if (index < 0 || index >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
      p = ctx->ext_count[index]; n = E; break;
    case AOM_B_SLOPES: p = ctx->slopes; n = E * ctx->lds; break;
    case AOM_B_ERR: p = ctx->err_v; n = E * ctx->lda; break;
    case AOM_B_COM: p = ctx->com; n = E * ctx->lda; break;
    case AOM_B_VOLTS: p = ctx->volts; n = E * ctx->lda; break;
    case AOM_B_BINCUBE:
      if (!ctx->bincube) CU(dalloc(&ctx->bincube, E * c.nvalid * 256));
      p = ctx->bincube; n = E * c.nvalid * 256; break;
    case AOM_B_PHASE:
      if (!ctx->phase) CU(dalloc(&ctx->phase, E * c.n * c.n));
      p = ctx->phase; n = E * c.n * c.n; break;
    case AOM_B_MODES: p = ctx->modes; n = E * ctx->ldm; break;
    case AOM_B_RES_MODES: p = ctx->modes_res; n = E * ctx->ldm; break;
    case AOM_B_STATE: p = ctx->state; n = E * ctx->ldst; break;
    case AOM_B_REWARD: p = ctx->reward; n = E * c.n_agents; break;
    case AOM_B_ACTION: p = ctx->action; n = E * ctx->ldact; break;
    case AOM_B_ACTION_MEAN: p = ctx->action_mean; n = E * ctx->ldact; break;
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
static int launch_gemm(aom_ctx* ctx, int epi, const float* A, int lda, long long sA, const float* B, int ldb,
                       long long sB, float* C, int ldc, long long sC, int M, int N, int K, const float* bias,
                       long long sBias, int relu, int batch, cudaStream_t st, float* com = nullptr, int ldcom = 0,
                       bool exact = false, const float* Bt = nullptr, long long sBt = 0) {
  GemmParams p;
  memset(&p, 0, sizeof(p));
  int Kp = AOM_LD(K);
  if (lda < Kp || ldb < Kp || (lda & 3) || (ldb & 3) || (ldc & 3) || ldc < N)
    return fail(ctx, AOM_ERR_INVALID, "gemm: leading dimensions must cover K rounded to 16 (lda %d ldb %d ldc %d K %d N %d)", lda, ldb, ldc, K, N);
  p.A = A; p.B = B; p.C = C; p.bias = bias;
  p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.M = M; p.N = N; p.K = Kp;
  p.sA = sA; p.sB = sB; p.sC = sC; p.sBias = sBias; p.relu = relu;
  p.com = com; p.ldcom = ldcom; p.gain = ctx->gain; p.closed = ctx->closed;
  p.Bt = Bt; p.sBt = sBt;
  if (epi == 1 && ctx->gain_env) { epi = 2; p.gain_env = ctx->gain_env; }   // integrator with one gain per environment
  // `exact`: float32 FFMA accumulation with round-to-nearest (the recursive screen extrusion needs it: the
  // tensor core truncates its float32 accumulator, a ~1e-5 systematic shrink that an autoregression integrates)
  if (!exact && ctx->opt[AOM_OPT_GEMM_PATH] != AOM_GEMM_SIMT) {
    // column tile: the wide one when it saves CTA waves (two CTAs per SM)
    const long long slots = 2LL * ctx->num_sms, rows = (M + GTC_BM - 1) / GTC_BM;
    auto waves = [&](int bn) { return (double)((rows * ((ldc + bn - 1) / bn) * batch + slots - 1) / slots) * bn; };
    const int bn = (!Bt && waves(GTC_BN_WIDE) < waves(GTC_BN)) ? GTC_BN_WIDE : GTC_BN;
    const dim3 grid((ldc + bn - 1) / bn, (unsigned)rows, batch);
    gemm_tc_each([&](auto kernel, size_t smem, int e, int b) {
      if (e == epi && b == bn) kernel<<<grid, GTC_THREADS, smem, st>>>(p, ctx->d_err);
    });
  } else if (exact && epi == 0 && batch == 1 && !bias && !relu && ctx->opt[AOM_OPT_GEMM_PATH] != AOM_GEMM_SIMT) {
    // shaped exact kernel: column tile 8 CN with the least padding.  Only columns < N are consumed by the
    // extrusion scatter; pad columns inside the last tile are written as zeros, the rest keep their zeros.
    int best = 9, waste = 1 << 30;
    for (int cn = 9; cn >= 8; --cn) {
      const int bn = 8 * cn, w = (N + bn - 1) / bn * bn - N;
      if (w < waste) { waste = w; best = cn; }
    }
    const int bn = 8 * best;
    // two K halves per tile when the tiles alone leave the SMs at two CTAs (8 warps) each
    const int tiles = ((N + bn - 1) / bn) * ((M + GEMM_BM - 1) / GEMM_BM);
    const int ksplit = (tiles <= 2 * ctx->num_sms && K >= 512) ? 2 : 1;
    if (ksplit > 1) {
      cudaError_t e = cudaMemsetAsync(C, 0, (size_t)M * ldc * sizeof(float), st);
      if (e != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    }
    dim3 grid((N + bn - 1) / bn, (M + GEMM_BM - 1) / GEMM_BM, ksplit);
    with<8, 9>(best, [&](auto CN) { gemm_tn_exact_kernel<CN><<<grid, 128, 0, st>>>(p); });
  } else {
    dim3 grid((ldc + GEMM_BN - 1) / GEMM_BN, (M + GEMM_BM - 1) / GEMM_BM, batch);
    with<0, 1, 2>(epi, [&](auto EPI) { gemm_tn_kernel<EPI><<<grid, 256, 0, st>>>(p); });
  }
  KCHECK();
  return AOM_OK;
}

// out[E][ldo] = X[E][ldx] . OP^T with the operator's digit planes (table id `op`): exact integer accumulation, one
// rounding to float32 -- the oracle's float64 evaluation of the controller products (oracle/loop.py)
static int launch_oz_product(aom_ctx* ctx, int op, const float* X, int ldx, int K, float* out, int ldo, int N, int integrator,
                             float* com, int ldcom, cudaStream_t st) {
  const aom_config& c = ctx->cfg;
  const int KB = ctx->ozop_kb[op], NT = ctx->ozop_nt[op], MT = (c.n_env + OZ_BM - 1) / OZ_BM;
  const size_t need = (size_t)MT * KB * OZ_SLICES * OZ_A_TILE;
  if (need > ctx->oz_xs_bytes) {
    cudaFree(ctx->oz_xs); ctx->oz_xs = nullptr; ctx->oz_xs_bytes = 0;
    CU(cudaMalloc((void**)&ctx->oz_xs, need));
    CU(cudaMemsetAsync(ctx->oz_xs, 0, need, st));
    ctx->oz_xs_bytes = need;
  }
  if (!ctx->oz_xev) CU(dalloc(&ctx->oz_xev, (size_t)c.n_env));
  OzSliceParams sl;
  sl.X = X; sl.ld = ldx; sl.K = K; sl.E = c.n_env; sl.KB = KB; sl.Zs = ctx->oz_xs; sl.ev = ctx->oz_xev;
  OzGemmParams m;
  memset(&m, 0, sizeof(m));
  m.Zs = ctx->oz_xs; m.ABs = ctx->ozop[op]; m.ev = ctx->oz_xev; m.ea = ctx->ozop_ea[op]; m.out = out; m.ldo = ldo;
  m.E = c.n_env; m.N = N; m.KB = KB; m.com = com; m.ldcom = ldcom; m.gain = ctx->gain; m.closed = ctx->closed; m.err = ctx->d_err;
  m.gain_env = integrator ? ctx->gain_env : nullptr;
  cudaError_t le = oz_product_launch(sl, m, integrator, MT, NT, st);
  if (le != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "oz_product_launch: %s", cudaGetErrorString(le));
  ctx->launches += 2;
  return AOM_OK;
}

extern "C" int aom_gemm_tn(aom_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                           int M, int N, int K, const float* bias, int relu, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  return launch_gemm(ctx, 0, A, lda, 0, B, ldb, 0, C, ldc, 0, M, N, K, bias, 0, relu, 1, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// steps != null: per-environment winds -- pass `pass` of the signed counts steps [E] of this axis (`sign` unused).
// envs != null: only the K environments envs[0..K) (device), compacted into the first K rows of the scratch and the
// contraction (the start-up of aom_reset_envs).
static int extrude_once(aom_ctx* ctx, int l, int axis, int sign, cudaStream_t st, const int* steps = nullptr, int pass = 0,
                        const int* envs = nullptr, int K = 0) {
  const aom_config& c = ctx->cfg;
  const int rows = envs ? K : c.n_env;
  NEED(AOM_T_AB, l);
  NEED(AOM_T_STENCIL, l);
  ExtrudeParams p;
  p.screen = ctx->screen[l]; p.ox = ctx->ox[l]; p.oy = ctx->oy[l]; p.count = ctx->ext_count[l];
  p.k0 = ctx->k0; p.k1 = ctx->k1; p.stencil = (const int*)ctx->tab[AOM_T_STENCIL][l];
  p.N = c.screen_dim[l]; p.S = c.stencil_size[l]; p.E = c.n_env; p.layer = l; p.axis = axis; p.sign = sign;
  p.amp = c.amp[l]; p.amp_env = ctx->amp_env[l];
  p.ldz = AOM_LD(p.S + p.N); p.Z = ctx->Z; p.zref = ctx->zref; p.ldn = AOM_LD(p.N); p.newcol = ctx->newcol;
  p.steps = steps; p.pass = pass; p.envs = envs;
  if (ctx->opt[AOM_OPT_EXTRUDE_PATH] == AOM_EXTRUDE_I8) {
    // exact integer contraction on tcgen05 (extrude_i8.cuh): digits of the inputs, 13 int8 digit-pair products with
    // int32 accumulators, one rounding to float32 after adding the reference pixel
    const int KB = ctx->oz_kb[l], NT = ctx->oz_nt[l], MT = (rows + OZ_BM - 1) / OZ_BM;
    const size_t need = (size_t)MT * KB * OZ_SLICES * OZ_A_TILE;
    if (need > ctx->oz_zs_bytes) {
      cudaFree(ctx->oz_zs); ctx->oz_zs = nullptr; ctx->oz_zs_bytes = 0;
      CU(cudaMalloc((void**)&ctx->oz_zs, need));
      CU(cudaMemsetAsync(ctx->oz_zs, 0, need, st));      // on the consuming stream: a default-stream memset does not order with it
      ctx->oz_zs_bytes = need;
    }
    if (!ctx->oz_ev) CU(dalloc(&ctx->oz_ev, (size_t)c.n_env));
    uint8_t* zs = ctx->oz_zs;
    int* ev = ctx->oz_ev;
    OzGatherParams g;
    g.screen = p.screen; g.ox = p.ox; g.oy = p.oy; g.count = p.count; g.k0 = p.k0; g.k1 = p.k1; g.stencil = p.stencil;
    g.zref = p.zref; g.ev = ev; g.Zs = zs; g.N = p.N; g.S = p.S; g.E = rows; g.KB = KB; g.layer = l;
    g.axis = axis; g.sign = sign; g.amp = p.amp; g.amp_env = ctx->amp_env[l];
    g.steps = steps; g.pass = pass; g.envs = envs;
    OzGemmParams m;
    m.Zs = zs; m.ABs = ctx->oz_ab[l]; m.ev = ev; m.ea = ctx->oz_ea[l]; m.zref = p.zref;
    m.out = p.newcol; m.ldo = p.ldn; m.E = rows; m.N = p.N; m.KB = KB; m.err = ctx->d_err;
    cudaError_t le = oz_extrude_launch(g, m, MT, NT, st);
    if (le != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "oz_extrude_launch: %s", cudaGetErrorString(le));
    ctx->launches += 2;
    p.zref = nullptr;                                  // the reference pixel is already in the new column
  } else {
    with<false, true>(steps != nullptr, [&](auto PE) { extrude_gather_kernel<PE><<<rows, 256, 0, st>>>(p); });
    KCHECK();
    int rc = launch_gemm(ctx, 0, ctx->Z, p.ldz, 0, (const float*)ctx->tab[AOM_T_AB][l], p.ldz, 0, ctx->newcol, p.ldn, 0,
                         rows, p.N, p.S + p.N, nullptr, 0, 0, 1, st, nullptr, 0, true);
    if (rc) return rc;
  }
  with<false, true>(steps != nullptr, [&](auto PE) { extrude_scatter_kernel<PE><<<rows, EXTRUDE_SCATTER_THREADS, 0, st>>>(p); });
  KCHECK();
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// per-environment winds
static bool wind_any_env(const aom_ctx* ctx) {
  for (int l = 0; l < ctx->cfg.n_layers; ++l)
    if (ctx->wind_dx[l]) return true;
  return false;
}

// One transition of the wind state of every layer and environment (WIND_STEP / WIND_INIT / WIND_RESET, atmos_kernels.cuh)
// on the device, asynchronously on `st`, and the same on the host mirror: passes per layer and offset bounds.
// WIND_RESET_ENVS: WIND_RESET of the K environments listed in envs_d (device) / envs_h (host) only.
static int wind_update(aom_ctx* ctx, int mode, cudaStream_t st, const int* envs_d = nullptr, const int* envs_h = nullptr,
                       int K = 0) {
  const aom_config& c = ctx->cfg;
  const int E = c.n_env, L = c.n_layers;
  if (L == 0) return AOM_OK;
  WindStateParams P;
  memset(&P, 0, sizeof(P));
  for (int l = 0; l < L; ++l) {
    WindLayerParams& W = P.layer[l];
    W.dx = ctx->wind_dx[l]; W.dy = ctx->wind_dy[l]; W.cdx = c.deltax[l]; W.cdy = c.deltay[l];
    W.ax0 = ctx->accx[l]; W.ay0 = ctx->accy[l]; W.xoff = c.wfs_xoff[l]; W.yoff = c.wfs_yoff[l]; W.n2 = 2 * c.screen_dim[l];
  }
  P.acc = ctx->wind_acc; P.steps = ctx->wind_steps; P.rec = ctx->wind_rec; P.E = E; P.n_layers = L; P.mode = mode;
  P.envs = envs_d; P.K = K;
  const int n = mode == WIND_RESET_ENVS ? K : E;
  wind_state_kernel<<<(L * n + 255) / 256, 256, 0, st>>>(P);
  KCHECK();
  for (int l = 0; l < L; ++l) {
    const WindLayerParams& W = P.layer[l];
    double* ax = ctx->wind_hacc + (size_t)2 * l * E;
    double* ay = ax + E;
    int px = 0, py = 0;
    int* box = ctx->wind_box[l];
    if (mode == WIND_RESET_ENVS) {
      for (int k = 0; k < K; ++k) ax[envs_h[k]] = ay[envs_h[k]] = 0.0;
      py = W.n2;
    }
    for (int e = 0; e < E; ++e) {
      const float dx = ctx->wind_hdx[l] ? ctx->wind_hdx[l][e] : W.cdx, dy = ctx->wind_hdy[l] ? ctx->wind_hdy[l][e] : W.cdy;
      if (mode == WIND_STEP) {
        const int nx = wind_advance(ax[e], dx), ny = wind_advance(ay[e], dy);
        px = std::max(px, abs(nx)); py = std::max(py, abs(ny));
      } else if (mode == WIND_INIT) {
        ax[e] = W.ax0; ay[e] = W.ay0;
      } else if (mode == WIND_RESET) {
        ax[e] = ay[e] = 0.0;
        py = W.n2;
      }
      const WindRec r = wind_record(W.xoff, W.yoff, ax[e], ay[e]);
      if (e == 0 || r.ix < box[0]) box[0] = r.ix;
      if (e == 0 || r.ix > box[1]) box[1] = r.ix;
      if (e == 0 || r.iy < box[2]) box[2] = r.iy;
      if (e == 0 || r.iy > box[3]) box[3] = r.iy;
    }
    ctx->wind_passes[l][0] = px; ctx->wind_passes[l][1] = py;
  }
  return AOM_OK;
}

// Back to the common accumulators once no layer has winds of its own and every layer's accumulators agree over the batch
// (at the latest after the next aom_reset, which zeroes them): the uniform kernels then run again.
static void wind_try_uniform(aom_ctx* ctx) {
  if (!ctx->wind_pe || wind_any_env(ctx)) return;
  const int E = ctx->cfg.n_env;
  for (int l = 0; l < ctx->cfg.n_layers; ++l) {
    const double* a = ctx->wind_hacc + (size_t)2 * l * E;
    for (int e = 1; e < E; ++e)
      if (a[e] != a[0] || a[E + e] != a[E]) return;
  }
  for (int l = 0; l < ctx->cfg.n_layers; ++l) {
    ctx->accx[l] = ctx->wind_hacc[(size_t)2 * l * E];
    ctx->accy[l] = ctx->wind_hacc[(size_t)(2 * l + 1) * E];
  }
  ctx->wind_pe = false;
}

// Per-environment wind state from the common one (WIND_INIT on `st`): every environment continues from the layer's
// common accumulators.
static int wind_begin_pe(aom_ctx* ctx, cudaStream_t st) {
  const size_t LE = (size_t)ctx->cfg.n_layers * ctx->cfg.n_env;
  if (!ctx->wind_acc) {
    CU(dalloc(&ctx->wind_acc, 2 * LE));
    CU(dalloc(&ctx->wind_steps, 2 * LE));
    CU(cudaMalloc((void**)&ctx->wind_rec, LE * sizeof(WindRec)));
    ctx->wind_hacc = (double*)calloc(2 * LE, sizeof(double));
    if (!ctx->wind_hacc) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
  }
  int rc = wind_update(ctx, WIND_INIT, st);
  if (rc) return rc;
  ctx->wind_pe = true;
  return AOM_OK;
}

extern "C" int aom_set_layer_wind(aom_ctx* ctx, int layer, const float* deltax_host, const float* deltay_host) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  if (layer < 0 || layer >= c.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
  if (!deltax_host != !deltay_host) return fail(ctx, AOM_ERR_INVALID, "per-environment winds need both components (or neither)");
  const size_t E = c.n_env;
  CU(cudaDeviceSynchronize());                       // an extrusion in flight may still read the old steps
  if (!deltax_host) {
    cudaFree(ctx->wind_dx[layer]); cudaFree(ctx->wind_dy[layer]); free(ctx->wind_hdx[layer]); free(ctx->wind_hdy[layer]);
    ctx->wind_dx[layer] = ctx->wind_dy[layer] = ctx->wind_hdx[layer] = ctx->wind_hdy[layer] = nullptr;
    wind_try_uniform(ctx);
    return AOM_OK;
  }
  for (size_t e = 0; e < E; ++e)
    if (!isfinite(deltax_host[e]) || !isfinite(deltay_host[e]))
      return fail(ctx, AOM_ERR_INVALID, "layer %d: wind of environment %zu is not finite", layer, e);
  if (!ctx->wind_hdx[layer]) {
    ctx->wind_hdx[layer] = (float*)malloc(E * sizeof(float));
    ctx->wind_hdy[layer] = (float*)malloc(E * sizeof(float));
    if (!ctx->wind_hdx[layer] || !ctx->wind_hdy[layer]) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    CU(cudaMalloc((void**)&ctx->wind_dx[layer], E * sizeof(float)));
    CU(cudaMalloc((void**)&ctx->wind_dy[layer], E * sizeof(float)));
  }
  memcpy(ctx->wind_hdx[layer], deltax_host, E * sizeof(float));
  memcpy(ctx->wind_hdy[layer], deltay_host, E * sizeof(float));
  CU(cudaMemcpy(ctx->wind_dx[layer], deltax_host, E * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ctx->wind_dy[layer], deltay_host, E * sizeof(float), cudaMemcpyHostToDevice));
  if (!ctx->wind_pe) {
    // every environment continues from the common accumulators: the screens do not jump
    int rc = wind_begin_pe(ctx, 0);
    if (rc) return rc;
    CU(cudaStreamSynchronize(0));                    // the legacy stream: the state is read next on any stream
  }
  const int* b = ctx->wind_box[layer];
  if (b[0] < 0 || b[2] < 0 || b[1] + c.n + 1 > c.screen_dim[layer] || b[3] + c.n + 1 > c.screen_dim[layer])
    return fail(ctx, AOM_ERR_UNSUPPORTED, "layer %d: pupil footprint leaves the screen", layer);
  return AOM_OK;
}

extern "C" int aom_move_atmos(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_move_atmos");
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  if (ctx->wind_pe) {
    // per-environment winds: counts and offsets on the device, passes sized by the host mirror (x then y, as below);
    // an environment takes part in the first |count| passes of each axis
    int rc = wind_update(ctx, WIND_STEP, st);
    if (rc) return rc;
    const size_t E = c.n_env;
    for (int l = 0; l < c.n_layers; ++l)
      for (int a = 0; a < 2; ++a)
        for (int i = 0; i < ctx->wind_passes[l][a]; ++i) {
          rc = extrude_once(ctx, l, a, 1, st, ctx->wind_steps + (2 * l + a) * E, i);
          if (rc) return rc;
        }
    wind_try_uniform(ctx);
    return AOM_OK;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    ctx->accx[l] += (double)c.deltax[l];
    ctx->accy[l] += (double)c.deltay[l];
    int nx = (int)ctx->accx[l], ny = (int)ctx->accy[l];
    ctx->accx[l] -= nx;
    ctx->accy[l] -= ny;
    for (int i = 0; i < abs(nx); ++i) { int rc = extrude_once(ctx, l, 0, nx > 0 ? 1 : -1, st); if (rc) return rc; }
    for (int i = 0; i < abs(ny); ++i) { int rc = extrude_once(ctx, l, 1, ny > 0 ? 1 : -1, st); if (rc) return rc; }
  }
  return AOM_OK;
}

static int clear_loop_state(aom_ctx* ctx, cudaStream_t st) {
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  CU(cudaMemsetAsync(ctx->slopes, 0, E * ctx->lds * 4, st));
  CU(cudaMemsetAsync(ctx->slopes_frame, 0, E * ctx->lds * 4, st));
  CU(cudaMemsetAsync(ctx->err_v, 0, E * ctx->lda * 4, st));
  CU(cudaMemsetAsync(ctx->com, 0, E * ctx->lda * 4, st));
  CU(cudaMemsetAsync(ctx->com1, 0, E * ctx->lda * 4, st));
  CU(cudaMemsetAsync(ctx->volts, 0, E * ctx->lda * 4, st));
  CU(cudaMemsetAsync(ctx->com_before, 0, E * ctx->lda * 4, st));
  if (ctx->modes_res) CU(cudaMemsetAsync(ctx->modes_res, 0, E * ctx->ldm * 4, st));
  if (ctx->hist) CU(cudaMemsetAsync(ctx->hist, 0, (size_t)c.n_hist * E * c.state_modes * 4, st));
  if (ctx->state) CU(cudaMemsetAsync(ctx->state, 0, E * ctx->ldst * 4, st));
  if (ctx->action) CU(cudaMemsetAsync(ctx->action, 0, E * ctx->ldact * 4, st));
  ctx->hist_head = 0;
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

static int start_screens(aom_ctx* ctx, const int* envs, int K, cudaStream_t st);

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
  for (int l = 0; l < c.n_layers; ++l) ctx->accx[l] = ctx->accy[l] = 0.0;
  if (ctx->wind_pe && !wind_any_env(ctx)) ctx->wind_pe = false;      // every accumulator restarts from 0: common again
  if (ctx->wind_pe) {
    // per-environment winds: accumulators 0, start-up counts 2N along y signed like each environment's x wind
    rc = wind_update(ctx, WIND_RESET, st);
    if (rc) return rc;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    size_t N = c.screen_dim[l];
    CU(cudaMemsetAsync(ctx->screen[l], 0, E * N * N * 4, st));
    CU(cudaMemsetAsync(ctx->ox[l], 0, E * 4, st));
    CU(cudaMemsetAsync(ctx->oy[l], 0, E * 4, st));
    CU(cudaMemsetAsync(ctx->ext_count[l], 0, E * 4, st));
  }
  return start_screens(ctx, nullptr, 0, st);
}

// Start-up of the screens of every environment (envs null) or of the K environments envs[0..K) (device list, compacted
// extrusions): zero screens, ring origins and counters are expected, and the wind state of WIND_RESET (WIND_RESET_ENVS).
// (The layers' start-up chains are independent, but running them on separate streams with private scratch gained
// nothing for the whole batch -- 1.35 s either way at 4096 environments: every extrusion kernel fills the GPU by itself.)
static int start_screens(aom_ctx* ctx, const int* envs, int K, cudaStream_t st) {
  const aom_config& c = ctx->cfg;
  const size_t E = c.n_env;
  const unsigned rows = envs ? (unsigned)K : (unsigned)E;
  int rc;
  for (int l = 0; l < c.n_layers; ++l) {
    size_t N = c.screen_dim[l];
    int sign = c.deltax[l] < 0 ? -1 : 1;
    const int* steps = ctx->wind_pe ? ctx->wind_steps + (2 * l + 1) * E : nullptr;
    // The reference starts a screen with 2N extrusions along x (columns: 648 pixels in 648 different DRAM rows per
    // environment, the expensive direction of the [y][x] layout -- 0.32 ms per extrusion at 4096 environments against
    // 0.19 ms along y).  From a zero screen with zero ring offsets the recursion along y produces exactly the transpose
    // (same stencil, same operator, same innovation counters; every index expression of the gather / scatter swaps its
    // roles, atmos_kernels.cuh / extrude_i8.cuh), and 2N extrusions bring the ring origin back to zero: so the start-up
    // runs along y and the screens are transposed in place once at the end -- bit-identical pixels, 1.29 -> 0.8 s.
    for (size_t i = 0; i < 2 * N; ++i) { rc = extrude_once(ctx, l, 1, sign, st, steps, (int)i, envs, K); if (rc) return rc; }
    {
      const int T = (int)((N + 31) / 32);
      transpose_screens_kernel<<<dim3((unsigned)(T * (T + 1) / 2), rows), dim3(32, 8), 0, st>>>(ctx->screen[l], (int)N, envs);
      KCHECK();
      // ring origin: 2N steps along y leave oy = 0 as 2N steps along x leave ox = 0 (2N mod N); nothing to swap
    }
  }
  return AOM_OK;
}

extern "C" int aom_reset_envs(aom_ctx* ctx, int n, const int32_t* envs, const int64_t* seeds, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  const int E = c.n_env;
  if (n < 0) return fail(ctx, AOM_ERR_INVALID, "aom_reset_envs: negative environment count %d", n);
  if (n > 0 && (!envs || !seeds)) return fail(ctx, AOM_ERR_INVALID, "null argument");
  if (n > E) return fail(ctx, AOM_ERR_INVALID, "aom_reset_envs: %d environments listed, the batch has %d", n, E);
  {
    char* seen = (char*)calloc((size_t)E, 1);
    if (!seen) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    for (int k = 0; k < n; ++k) {
      const int e = envs[k];
      if (e < 0 || e >= E) { free(seen); return fail(ctx, AOM_ERR_INVALID, "aom_reset_envs: environment %d out of range [0, %d)", e, E); }
      if (seen[e]) { free(seen); return fail(ctx, AOM_ERR_INVALID, "aom_reset_envs: environment %d listed twice", e); }
      seen[e] = 1;
    }
    free(seen);
  }
  if (!ctx->seeded) return fail(ctx, AOM_ERR_STATE, "aom_reset must be called before aom_reset_envs");
  if (n == 0) return AOM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CU(cudaStreamSynchronize(st));                     // the wind mirror and the staging buffers are updated from the host
  if (!ctx->first) {
    CU(dalloc(&ctx->rs_envs, (size_t)E));
    CU(dalloc(&ctx->rs_seeds, 2 * (size_t)E));
    CU(dalloc(&ctx->frame0, (size_t)E));
    CU(dalloc(&ctx->step_env, (size_t)E));
    CU(dalloc(&ctx->le_n, 2 * (size_t)E));
    CU(dalloc(&ctx->first, (size_t)E));
  }
  if (!ctx->staggered) {
    // the batch leaves lockstep: every environment's counters start at the batch's
    stagger_counters_kernel<<<(E + 255) / 256, 256, 0, st>>>(ctx->frame0, ctx->step_env, ctx->le_n, ctx->first, E, ctx->step,
                                                             ctx->tar_n, ctx->geo_tar_n);
    KCHECK();
    ctx->staggered = true;
  }
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
  auto add = [&](void* b, long long ld, int slots = 1, long long slot_stride = 0) {
    if (!b || P.nbuf == RESET_MAX_BUFS) return;
    P.buf[P.nbuf] = (uint32_t*)b; P.ld[P.nbuf] = ld; P.slots[P.nbuf] = slots; P.slot_stride[P.nbuf] = slot_stride;
    P.nbuf++;
  };
  add(ctx->slopes, ctx->lds); add(ctx->slopes_frame, ctx->lds); add(ctx->err_v, ctx->lda); add(ctx->com, ctx->lda);
  add(ctx->com1, ctx->lda); add(ctx->volts, ctx->lda); add(ctx->com_before, ctx->lda); add(ctx->modes_res, ctx->ldm);
  add(ctx->state, ctx->ldst); add(ctx->action, ctx->ldact); add(ctx->tar_acc, TAR_ACC); add(ctx->strehl, 4);
  if (ctx->hist) add(ctx->hist, c.state_modes, c.n_hist, (long long)E * c.state_modes);   // every slot of the ring
  add(ctx->geo_com, ctx->lda); add(ctx->geo_volts, ctx->lda); add(ctx->geo_acc, TAR_ACC); add(ctx->strehl_geo, 4);
  for (int l = 0; l < c.n_layers; ++l) {
    add(ctx->screen[l], (long long)c.screen_dim[l] * c.screen_dim[l]);
    add(ctx->ox[l], 1); add(ctx->oy[l], 1); add(ctx->ext_count[l], 1);
  }
  P.envs = ctx->rs_envs; P.seeds = ctx->rs_seeds; P.K = n; P.E = E;
  P.k0 = ctx->k0; P.k1 = ctx->k1; P.frame0 = ctx->frame0; P.step_env = ctx->step_env; P.le_n = ctx->le_n;
  P.first = ctx->first; P.frame = ctx->frame;
  reset_envs_kernel<<<dim3((unsigned)n, (unsigned)P.nbuf + 1), 256, 0, st>>>(P);
  KCHECK();
  ctx->first_any = true;
  if (c.n_layers == 0) return AOM_OK;
  // The listed environments' accumulators restart from 0 while the others keep theirs: the per-environment wind state
  // (common winds included) until they agree again (wind_try_uniform)
  int rc;
  if (!ctx->wind_pe) { rc = wind_begin_pe(ctx, st); if (rc) return rc; }
  rc = wind_update(ctx, WIND_RESET_ENVS, st, ctx->rs_envs, envs, n);
  if (rc) return rc;
  return start_screens(ctx, ctx->rs_envs, n, st);
}

// ---------------------------------------------------------------------------------------------
// Host side of the staged sensor kernels, wfs_frame_tma_kernel (wfs_tma.cuh) and the tcgen05 pair (wfs_umma.cuh,
// wfs_umma_ws.cuh): eligibility, derived tables, TMA descriptors.  Both read the mirror through the same lattice
// analysis (wfs_lattice_host.h) and lay out its tables their own way.
static uint32_t half2_bits(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  uint32_t u;
  memcpy(&u, &h, 4);
  return u;
}

static void split_pair(double a, double b, int lo_part, uint32_t& out) {
  const float ah = __half2float(__float2half_rn((float)a)), bh = __half2float(__float2half_rn((float)b));
  out = lo_part ? half2_bits((float)(a - (double)ah), (float)(b - (double)bh)) : half2_bits(ah, bh);
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

// A staged kernel cannot serve this configuration: its state becomes -1 and fast_why says why.  Returns AOM_OK.
static int staged_refuse(aom_ctx* ctx, int& state, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(ctx->fast_why, sizeof(ctx->fast_why), fmt, ap);
  va_end(ap);
  state = -1;
  return AOM_OK;
}

// The lattice analysis of the uploaded host tables: null, or why the staged kernels cannot serve them
static const char* staged_lattice(aom_ctx* ctx, WfsLattice& L) {
  return wfl_analyse(ctx->cfg, (const float*)ctx->htab[AOM_T_MPUPIL], (const int*)ctx->htab[AOM_T_SUB_X0],
                     (const int*)ctx->htab[AOM_T_SUB_Y0], (const float*)ctx->htab[AOM_T_STAMP1D],
                     (const int*)ctx->htab[AOM_T_ACT_MAP], L);
}

// One 3-D map [E][N][N] per screen layer, box bw x bh x 1, zero fill outside.  False: refused (state, fast_why).
static bool encode_screen_maps(aom_ctx* ctx, CUtensorMap* maps, cuuint32_t bw, cuuint32_t bh, int& state) {
  const aom_config& c = ctx->cfg;
  if (c.n_layers == 0) return true;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    staged_refuse(ctx, state, "cuTensorMapEncodeTiled not available");
    return false;
  }
  for (int l = 0; l < c.n_layers; ++l) {
    const cuuint64_t N = (cuuint64_t)c.screen_dim[l];
    const cuuint64_t dims[3] = {N, N, (cuuint64_t)c.n_env};
    const cuuint64_t strides[2] = {N * 4, N * N * 4};
    const cuuint32_t box[3] = {bw, bh, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = ((aom_encode_tiled_fn)fn)(&maps[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ctx->screen[l], dims, strides, box,
                                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      staged_refuse(ctx, state, "cuTensorMapEncodeTiled failed (%d)", (int)r);
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

static int wfs_fast_prepare(aom_ctx* ctx) {
  const aom_config& c = ctx->cfg;
  if (ctx->fast_state != 0) return AOM_OK;
  for (void*& b : ctx->fast_dev) { cudaFree(b); b = nullptr; }
  WfsLattice L;
  if (const char* why = staged_lattice(ctx, L)) return staged_refuse(ctx, ctx->fast_state, "%s", why);
  const float* pup = (const float*)ctx->htab[AOM_T_MPUPIL];
  const int* sx = (const int*)ctx->htab[AOM_T_SUB_X0];
  const int* sy = (const int*)ctx->htab[AOM_T_SUB_Y0];
  const float* stamp = (const float*)ctx->htab[AOM_T_STAMP1D];
  const int nv = c.nvalid, GW = L.GW;
  uint2* h_sub = (uint2*)malloc((size_t)nv * sizeof(uint2));
  unsigned char* h_pm = (unsigned char*)malloc((size_t)nv * 32);
  short* h_amap = (short*)malloc((size_t)GW * GW * sizeof(short));
  float h_fxy[2 * WFT_NG * 16];
  uint4* h_c1 = (uint4*)malloc(8 * 32 * sizeof(uint4));
  uint4* h_c2 = (uint4*)malloc(12 * 32 * sizeof(uint4));
  const bool ok = h_sub && h_pm && h_amap && h_c1 && h_c2;
  if (ok) {
    wfl_amap(c, L, (const int*)ctx->htab[AOM_T_ACT_MAP], h_amap);
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
                           8 * 32 * sizeof(uint4), 12 * 32 * sizeof(uint4), sizeof(h_fxy)};
  const cudaError_t ce = ok ? upload_tables(ctx->fast_dev, srcs, sizes) : cudaSuccess;
  free(h_sub); free(h_pm); free(h_amap); free(h_c1); free(h_c2);
  if (ce != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "wfs_fast_prepare: %s", cudaGetErrorString(ce));
  if (!ok) return staged_refuse(ctx, ctx->fast_state, "out of host memory");
  if (!encode_screen_maps(ctx, ctx->fast_maps, WFT_TILE_W, WFT_TILE_H, ctx->fast_state)) return AOM_OK;
  WfsFast& f = ctx->fast;
  f.sub = (const uint2*)ctx->fast_dev[0];
  f.amap = (const short*)ctx->fast_dev[1];
  f.pmask = (const unsigned char*)ctx->fast_dev[2];
  f.c1 = (const uint4*)ctx->fast_dev[3];
  f.c2 = (const uint4*)ctx->fast_dev[4];
  f.fxy = (const float*)ctx->fast_dev[5];
  f.GW = GW;
  f.sub_in_smem = (nv <= 1280) ? 1 : 0;
  f.err = ctx->d_err;
  ctx->fast_state = 1;
  return AOM_OK;
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
static int wfs_umma_prepare(aom_ctx* ctx) {
  const aom_config& c = ctx->cfg;
  if (ctx->umma_state != 0) return AOM_OK;
  for (void*& b : ctx->umma_dev) { cudaFree(b); b = nullptr; }
  WfsLattice L;
  if (const char* why = staged_lattice(ctx, L)) return staged_refuse(ctx, ctx->umma_state, "%s", why);
  if (c.nvalid < WU_WARPS) return staged_refuse(ctx, ctx->umma_state, "fewer than %d subapertures", WU_WARPS);
  const float* hxy = (const float*)ctx->htab[AOM_T_HALFXY];
  if (!hxy) return staged_refuse(ctx, ctx->umma_state, "half-pixel phasor table not uploaded");
  for (int i = 0; i < 16; ++i)
    for (int j = 0; j < 16; ++j)
      if (fabs((double)hxy[i * 16 + j] - M_PI * (double)(i + j) / 64.0) > 2e-6)
        return staged_refuse(ctx, ctx->umma_state, "half-pixel phasor is not pi (x + y) / Nfft");
  const float* pup = (const float*)ctx->htab[AOM_T_MPUPIL];
  const int* sx = (const int*)ctx->htab[AOM_T_SUB_X0];
  const int* sy = (const int*)ctx->htab[AOM_T_SUB_Y0];
  const float* stamp = (const float*)ctx->htab[AOM_T_STAMP1D];
  const int nv = c.nvalid, GW = L.GW;
  uint2* h_sub = (uint2*)malloc((size_t)nv * sizeof(uint2));
  uint32_t* h_pm = (uint32_t*)malloc((size_t)nv * 32 * sizeof(uint32_t));
  short* h_amap = (short*)malloc((size_t)GW * GW * sizeof(short));
  unsigned short* h_b1 = (unsigned short*)calloc(2 * WU_B_BYTES, 1);     // [hi, lo] tiles of WU_B_BYTES each
  unsigned short* h_b2 = (unsigned short*)calloc(2 * WU_B_BYTES, 1);
  float h_fxy[2 * WU_NG * 16];
  const bool ok = h_sub && h_pm && h_amap && h_b1 && h_b2;
  if (ok) {
    wfl_amap(c, L, (const int*)ctx->htab[AOM_T_ACT_MAP], h_amap);
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
                           (size_t)2 * WU_B_BYTES, (size_t)2 * WU_B_BYTES, sizeof(h_fxy)};
  const cudaError_t ce = ok ? upload_tables(ctx->umma_dev, srcs, sizes) : cudaSuccess;
  free(h_sub); free(h_pm); free(h_amap); free(h_b1); free(h_b2);
  if (ce != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "wfs_umma_prepare: %s", cudaGetErrorString(ce));
  if (!ok) return staged_refuse(ctx, ctx->umma_state, "out of host memory");
  if (!encode_screen_maps(ctx, ctx->umma.maps, WU_TILE_W, WU_TILE_H, ctx->umma_state)) return AOM_OK;
  WfsUmmaTables& f = ctx->umma.f;
  memset(&f, 0, sizeof(f));
  f.sub = (const uint2*)ctx->umma_dev[0];
  f.amap = (const short*)ctx->umma_dev[1];
  f.pmask = (const uint32_t*)ctx->umma_dev[2];
  f.b1 = (const uint4*)ctx->umma_dev[3];
  f.b2 = (const uint4*)ctx->umma_dev[4];
  f.fxy = (const float*)ctx->umma_dev[5];
  f.GW = GW;
  f.err = ctx->d_err;
  ctx->umma_state = 1;
  return AOM_OK;
}

template <int FULL, int NL>
static int wfs_fast_launch_t(aom_ctx* ctx, const WfsParams& p, cudaStream_t st) {
  const long long total = (long long)p.E * p.nvalid;
  // contiguous ranges of work items per CTA: about 8 waves of resident CTAs per SM, at least 16 items per warp
  long long grid = (long long)ctx->num_sms * WFT_MIN_CTAS * 8;
  long long ipc = (total + grid - 1) / grid;
  if (ipc < 16 * WFT_WARPS) ipc = 16 * WFT_WARPS;
  ipc = (ipc + WFT_WARPS - 1) / WFT_WARPS * WFT_WARPS;
  grid = (total + ipc - 1) / ipc;
  WfsTmaParams P;
  memset(&P, 0, sizeof(P));
  P.p = p;
  P.f = ctx->fast;
  P.f.items_per_cta = ipc;
  for (int l = 0; l < NL; ++l) P.maps[l] = ctx->fast_maps[l];
  const size_t smem = wft_smem_bytes<NL>(P.f.GW, P.f.sub_in_smem ? p.nvalid : 0);
  {
    cudaError_t e = cudaFuncSetAttribute(wfs_frame_tma_kernel<FULL, NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "cudaFuncSetAttribute(wfs_frame_tma_kernel): %s", cudaGetErrorString(e));
  }
  wfs_frame_tma_kernel<FULL, NL><<<(unsigned)grid, WFT_WARPS * 32, smem, st>>>(P);
  return AOM_OK;
}

static int wfs_fast_launch(aom_ctx* ctx, const WfsParams& p, bool full, cudaStream_t st) {
  int rc = AOM_OK;
  const bool served = with<0, 1, 2, 3, 4>(p.n_layers, [&](auto NL) {
    with<false, true>(full, [&](auto FULL) { rc = wfs_fast_launch_t<FULL, NL>(ctx, p, st); });
  });
  return served ? rc : fail(ctx, AOM_ERR_UNSUPPORTED, "wfs_fast_launch: %d layers", p.n_layers);
}

// ---------------------------------------------------------------------------------------------
static int fill_wfs_params(aom_ctx* ctx, WfsParams& p, int flags, float noise) {
  const aom_config& c = ctx->cfg;
  memset(&p, 0, sizeof(p));
  NEED(AOM_T_MPUPIL, 0); NEED(AOM_T_HALFXY, 0); NEED(AOM_T_SUB_X0, 0); NEED(AOM_T_SUB_Y0, 0); NEED(AOM_T_FLUX, 0);
  p.n_layers = (flags & 1) ? c.n_layers : 0;
  for (int l = 0; l < p.n_layers; ++l) {
    WfsLayer& L = p.layer[l];
    L.screen = ctx->screen[l]; L.ox = ctx->ox[l]; L.oy = ctx->oy[l]; L.N = c.screen_dim[l];
    const WindRec r = wind_record(c.wfs_xoff[l], c.wfs_yoff[l], ctx->accx[l], ctx->accy[l]);
    L.ix = r.ix; L.iy = r.iy; L.fx = r.fx; L.fy = r.fy; L.w00 = r.w00; L.w01 = r.w01; L.w10 = r.w10; L.w11 = r.w11;
    int box[4] = {L.ix, L.ix, L.iy, L.iy};          // with per-environment winds: the extremes over the batch
    if (ctx->wind_pe) memcpy(box, ctx->wind_box[l], sizeof(box));
    if (box[0] < 0 || box[2] < 0 || box[1] + c.n + 1 > L.N || box[3] + c.n + 1 > L.N)
      return fail(ctx, AOM_ERR_UNSUPPORTED, "layer %d: pupil footprint leaves the screen", l);
  }
  p.wind = (ctx->wind_pe && p.n_layers > 0) ? ctx->wind_rec : nullptr;
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
  p.volts = ctx->volts; p.ldv = ctx->lda;
  p.stamp1d = (const float*)ctx->tab[AOM_T_STAMP1D][0]; p.ss = c.stamp_size;
  p.act_map = (const int*)ctx->tab[AOM_T_ACT_MAP][0];
  p.grid_n = c.pzt_grid_n; p.pitch = c.pzt_pitch; p.i1_0 = c.pzt_i1_0; p.j1_0 = c.pzt_j1_0;
  p.pzt_off = c.pzt_off; p.pzt_nact = c.pzt_nact;
  p.tt_planes = (const float*)ctx->tab[AOM_T_TT_PLANES][0]; p.tt_dim = c.tt_dim; p.tt_off = c.tt_off;
  p.k2 = (float)(2.0 * M_PI / (double)c.lambda_um);
  p.nphotons = ctx->nph_c; p.noise = noise; p.cog_offset = c.cog_offset; p.pixsize = c.pixsize;
  // per-environment sensor values: every frame is scaled by each environment's photon count, a noisy frame (noise >= 0)
  // draws each environment's own noise, a noise-free one none
  p.nph_env = ctx->nph_env;
  p.noise_env = (noise >= 0.f) ? ctx->noise_env : nullptr;
  p.frame = ctx->frame; p.wfs_index = (uint32_t)c.wfs_index; p.k0 = ctx->k0; p.k1 = ctx->k1;
  p.frame0 = ctx->staggered ? ctx->frame0 : nullptr;
  p.slopes = ctx->slopes_frame; p.lds = ctx->lds;
  return AOM_OK;
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

// Routes a frame of parameters p (fill_wfs_params), noisy when any environment draws noise in it, with its image kept or
// not.  Prepares the tables of a staged kernel on first use, and the round-1 kernel's only when the route can reach it.
static int wfs_route(aom_ctx* ctx, const WfsParams& p, bool noisy, bool keep, WfsRoute& r) {
  const aom_config& c = ctx->cfg;
  const int path = ctx->opt[AOM_OPT_WFS_PATH];
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
    int rc = wfs_umma_prepare(ctx);
    if (rc) return rc;
  }
  if (umma && ctx->umma_state == 1) {
    // the specialised-warp kernel serves every frame without noise and kept image (it reads neither noise nor photon
    // count); the others go to the fused kernel, in its per-environment form when per-environment values are in force
    r.family = (path == AOM_WFS_UMMA_WS && !noisy && !keep) ? WFS_WS : WFS_UMMA;
    if (r.family == WFS_WS) r.ne = false;
    return AOM_OK;
  }
  if (staged) {
    int rc = wfs_fast_prepare(ctx);
    if (rc) return rc;
  }
  r.family = (staged && ctx->fast_state == 1) ? WFS_TMA : WFS_MMA;
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
  bool noisy = p.noise >= 0.f;
  if (p.noise_env) {
    noisy = false;
    for (int e = 0; e < c.n_env && !noisy; ++e) noisy = ctx->noise_henv[e] >= 0.f;
  }
  WfsRoute r;
  rc = wfs_route(ctx, p, noisy, p.bincube != nullptr, r);
  if (rc) return rc;
  if (r.refused) return fail(ctx, AOM_ERR_UNSUPPORTED, "%s", r.refused);
  const bool timed = ctx->opt[AOM_OPT_TIME_WFS] && ctx->wev_n < AOM_WFS_TIMERS;
  if (timed) {
    for (int j = 0; j < 2; ++j)
      if (!ctx->wev[j][ctx->wev_n]) CU(cudaEventCreate(&ctx->wev[j][ctx->wev_n]));
    CU(cudaEventRecord(ctx->wev[0][ctx->wev_n], st));
  }
  long long total = (long long)c.n_env * c.nvalid;
  long long blocks = (total + WFS_WARPS - 1) / WFS_WARPS;
  long long cap = (long long)ctx->num_sms * 2 * 8;      // 2 resident CTAs per SM, 8 waves of work each
  int grid = (int)(blocks < cap ? blocks : cap);
  if (r.family == WFS_WS || r.family == WFS_UMMA) {
    if (r.family == WFS_WS) { p.noise = -1.f; p.noise_env = nullptr; p.nph_env = nullptr; }
    cudaError_t le = wfs_umma_launch(p, ctx->umma, ctx->num_sms, r.family == WFS_WS, r.full, r.ne, st);
    if (le != cudaSuccess) return fail(ctx, AOM_ERR_CUDA, "wfs_umma_launch: %s", cudaGetErrorString(le));
  } else if (r.family == WFS_TMA) {
    rc = wfs_fast_launch(ctx, p, r.full, st);
    if (rc) return rc;
  } else if (r.family == WFS_MMA) {
    with<0, 1, 3, -1>(r.nl, [&](auto NL) {
      with<false, true>(r.full, [&](auto FULL) { wfs_frame_mma_kernel<FULL, NL><<<grid, WFM_WARPS * 32, 0, st>>>(p); });
    });
  } else {
    wfs_simt_each([&](auto kernel, size_t smem, int R, bool PE, bool NE) {
      if (R == r.r && PE == r.pe && NE == r.ne) kernel<<<grid, WFS_WARPS * 32, smem, st>>>(p);
    });
  }
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
  // the route of a noise-free frame without kept image; the per-environment state does not change its family, so the
  // fields the route reads for it stay empty (and a refusal it would cause is not reported)
  const WfsParams p{};
  WfsRoute r;
  if (wfs_route(ctx, p, false, false, r) != AOM_OK) return "";
  if (r.family == WFS_MMA && ctx->opt[AOM_OPT_WFS_PATH] != AOM_WFS_MMA_REG)
    snprintf(ctx->err, sizeof(ctx->err), "staged sensor kernels not eligible: %s", ctx->fast_why);
  return wfs_kernel_names[r.family];
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
  return launch_gemm(ctx, 0, ctx->geo_b, ctx->lda, 0, (const float*)ctx->tab[AOM_T_GEO_PROJ][0], ctx->lda, 0, ctx->geo_com,
                     ctx->lda, 0, c.n_env, c.nactu, c.nactu, nullptr, 0, 0, 1, st, nullptr, 0, true);
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
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  NEED(AOM_T_CMAT, 0);
  if (ctx->opt[AOM_OPT_GEMM_PATH] == AOM_GEMM_TCGEN05 && ctx->ozop[AOM_T_CMAT])
    return launch_oz_product(ctx, AOM_T_CMAT, ctx->slopes, ctx->lds, c.nslopes, ctx->err_v, ctx->lda, c.nactu, 1, ctx->com,
                             ctx->lda, (cudaStream_t)stream);
  return launch_gemm(ctx, 1, ctx->slopes, ctx->lds, 0, (const float*)ctx->tab[AOM_T_CMAT][0], ctx->lds, 0, ctx->err_v,
                     ctx->lda, 0, c.n_env, c.nactu, c.nslopes, nullptr, 0, 0, 1, (cudaStream_t)stream, ctx->com, ctx->lda);
}

extern "C" int aom_set_command(aom_ctx* ctx, const float* dcom, int ld, void* stream) {
  if (!ctx || !dcom) return fail(ctx, AOM_ERR_INVALID, "null argument");
  const aom_config& c = ctx->cfg;
  if (ld < c.nactu) return fail(ctx, AOM_ERR_INVALID, "Dimension mismatch");
  dim3 grid((ctx->lda + 255) / 256, c.n_env);
  copy_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dcom, ld, ctx->com, ctx->lda, c.nactu, c.n_env);
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_set_dm_volts(aom_ctx* ctx, const float* dvolts, int ld, void* stream) {
  if (!ctx || !dvolts) return fail(ctx, AOM_ERR_INVALID, "null argument");
  const aom_config& c = ctx->cfg;
  if (ld < c.nactu) return fail(ctx, AOM_ERR_INVALID, "Dimension mismatch");
  dim3 grid((ctx->lda + 255) / 256, c.n_env);
  copy_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dvolts, ld, ctx->volts, ctx->lda, c.nactu, c.n_env);
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_apply_control(aom_ctx* ctx, int comp_voltage, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  size_t total = (size_t)c.n_env * ctx->lda;
  apply_control_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctx->com, ctx->com1, ctx->volts,
                                                                                         ctx->lda, total, c.delay, comp_voltage);
  KCHECK();
  return AOM_OK;
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
  if (!ctx) return AOM_ERR_INVALID;
  ctx->gain = gain;
  return AOM_OK;
}

// Per-environment value array: NULL frees it (back to the common value); otherwise checks every entry (finite, and > 0
// when `positive`), keeps a host copy and uploads it.  The caller has synchronised the device.
static int set_env_values(aom_ctx* ctx, const float* host, float** dev, float** hcopy, bool positive, const char* what) {
  const size_t E = ctx->cfg.n_env;
  if (!host) {
    cudaFree(*dev); free(*hcopy);
    *dev = *hcopy = nullptr;
    return AOM_OK;
  }
  for (size_t e = 0; e < E; ++e) {
    if (!isfinite(host[e])) return fail(ctx, AOM_ERR_INVALID, "%s of environment %zu is not finite", what, e);
    if (positive && !(host[e] > 0.f)) return fail(ctx, AOM_ERR_INVALID, "%s of environment %zu must be > 0", what, e);
  }
  if (!*hcopy) {
    *hcopy = (float*)malloc(E * sizeof(float));
    if (!*hcopy) return fail(ctx, AOM_ERR_INVALID, "out of host memory");
    CU(cudaMalloc((void**)dev, E * sizeof(float)));
  }
  memcpy(*hcopy, host, E * sizeof(float));
  CU(cudaMemcpy(*dev, host, E * sizeof(float), cudaMemcpyHostToDevice));
  return AOM_OK;
}

extern "C" int aom_set_gain_env(aom_ctx* ctx, const float* gain_host) {
  if (!ctx) return AOM_ERR_INVALID;
  CU(cudaDeviceSynchronize());                       // an integrator in flight may still read the old gains
  return set_env_values(ctx, gain_host, &ctx->gain_env, &ctx->gain_henv, false, "gain");
}

extern "C" int aom_set_wfs_noise(aom_ctx* ctx, float noise, float nphotons) {
  if (!ctx) return AOM_ERR_INVALID;
  if (!isfinite(noise) || !isfinite(nphotons)) return fail(ctx, AOM_ERR_INVALID, "sensor noise and photon count must be finite");
  if (!(nphotons > 0.f)) return fail(ctx, AOM_ERR_INVALID, "photon count must be > 0");
  ctx->noise_c = noise;
  ctx->nph_c = nphotons;
  return AOM_OK;
}

extern "C" int aom_set_wfs_noise_env(aom_ctx* ctx, const float* noise_host, const float* nphotons_host) {
  if (!ctx) return AOM_ERR_INVALID;
  const size_t E = ctx->cfg.n_env;
  // check both before changing either: a refused call leaves the state as it was
  for (size_t e = 0; noise_host && e < E; ++e)
    if (!isfinite(noise_host[e])) return fail(ctx, AOM_ERR_INVALID, "sensor noise of environment %zu is not finite", e);
  for (size_t e = 0; nphotons_host && e < E; ++e)
    if (!isfinite(nphotons_host[e]) || !(nphotons_host[e] > 0.f))
      return fail(ctx, AOM_ERR_INVALID, "photon count of environment %zu must be finite and > 0", e);
  CU(cudaDeviceSynchronize());                       // a sensor frame in flight may still read the old values
  int rc = set_env_values(ctx, noise_host, &ctx->noise_env, &ctx->noise_henv, false, "sensor noise");
  if (rc) return rc;
  return set_env_values(ctx, nphotons_host, &ctx->nph_env, &ctx->nph_henv, true, "photon count");
}

extern "C" int aom_set_loop(aom_ctx* ctx, int closed) {
  if (!ctx) return AOM_ERR_INVALID;
  ctx->closed = closed ? 1 : 0;
  return AOM_OK;
}

extern "C" int aom_set_layer(aom_ctx* ctx, int layer, float deltax, float deltay, float amp) {
  if (!ctx) return AOM_ERR_INVALID;
  if (layer < 0 || layer >= ctx->cfg.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
  ctx->cfg.deltax[layer] = deltax;
  ctx->cfg.deltay[layer] = deltay;
  ctx->cfg.amp[layer] = amp;
  return AOM_OK;
}

extern "C" int aom_set_layer_amp(aom_ctx* ctx, int layer, const float* amp_host) {
  if (!ctx) return AOM_ERR_INVALID;
  if (layer < 0 || layer >= ctx->cfg.n_layers) return fail(ctx, AOM_ERR_INVALID, "layer index out of range");
  if (!amp_host) { cudaFree(ctx->amp_env[layer]); ctx->amp_env[layer] = nullptr; return AOM_OK; }
  CU(cudaDeviceSynchronize());                       // an extrusion in flight may still read the old amplitudes
  if (!ctx->amp_env[layer]) CU(cudaMalloc((void**)&ctx->amp_env[layer], (size_t)ctx->cfg.n_env * sizeof(float)));
  CU(cudaMemcpy(ctx->amp_env[layer], amp_host, (size_t)ctx->cfg.n_env * sizeof(float), cudaMemcpyHostToDevice));
  return AOM_OK;
}

extern "C" int aom_reset_dm(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  CU(cudaMemsetAsync(ctx->volts, 0, (size_t)ctx->cfg.n_env * ctx->lda * 4, (cudaStream_t)stream));
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
static int project_v2m(aom_ctx* ctx, const float* v, float* out, cudaStream_t st) {
  const aom_config& c = ctx->cfg;
  NEED(AOM_T_V2M, 0);
  if (ctx->opt[AOM_OPT_GEMM_PATH] == AOM_GEMM_TCGEN05 && ctx->ozop[AOM_T_V2M])
    return launch_oz_product(ctx, AOM_T_V2M, v, ctx->lda, c.nactu, out, ctx->ldm, c.nmodes, 0, nullptr, 0, st);
  return launch_gemm(ctx, 0, v, ctx->lda, 0, (const float*)ctx->tab[AOM_T_V2M][0], ctx->lda, 0, out, ctx->ldm, 0, c.n_env,
                     c.nmodes, c.nactu, nullptr, 0, 0, 1, st);
}

extern "C" int aom_rl_control(aom_ctx* ctx, const float* daction, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  NEED(AOM_T_M2V, 0); NEED(AOM_T_FREEDOM, 0); NEED(AOM_T_ACTION_MAP, 0);
  const float* act = daction ? daction : ctx->action;
  if (!act) return fail(ctx, AOM_ERR_STATE, "no action buffer");
  int rc = project_v2m(ctx, ctx->com, ctx->modes, st);
  if (rc) return rc;
  dim3 grid((c.action_dim + 127) / 128, c.n_env);
  inject_action_kernel<<<grid, 128, 0, st>>>(ctx->modes, ctx->ldm, act, ctx->ldact, (const int*)ctx->tab[AOM_T_ACTION_MAP][0],
                                             (const float*)ctx->tab[AOM_T_FREEDOM][0], c.action_dim, c.n_env,
                                             c.env_act_scale, c.env_act_bias, ctx->first_any ? ctx->first : nullptr);
  KCHECK();
  if (ctx->opt[AOM_OPT_GEMM_PATH] == AOM_GEMM_TCGEN05 && ctx->ozop[AOM_T_M2V])
    return launch_oz_product(ctx, AOM_T_M2V, ctx->modes, ctx->ldm, c.nmodes, ctx->com, ctx->lda, c.nactu, 0, nullptr, 0, st);
  return launch_gemm(ctx, 0, ctx->modes, ctx->ldm, 0, (const float*)ctx->tab[AOM_T_M2V][0], ctx->ldm, 0, ctx->com, ctx->lda, 0,
                     c.n_env, c.nactu, c.nmodes, nullptr, 0, 0, 1, st);
}

extern "C" int aom_state_begin(aom_ctx* ctx, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  CU(cudaMemcpyAsync(ctx->com_before, ctx->com, (size_t)ctx->cfg.n_env * ctx->lda * 4, cudaMemcpyDeviceToDevice,
                     (cudaStream_t)stream));
  return AOM_OK;
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
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  if (!ctx->state) return fail(ctx, AOM_ERR_STATE, "state_dim is 0 in this configuration");
  NEED(AOM_T_STATE_MAP, 0); NEED(AOM_T_NORM_DM_MEAN, 0); NEED(AOM_T_NORM_DM_STD, 0);
  NEED(AOM_T_NORM_RES_MEAN, 0); NEED(AOM_T_NORM_RES_STD, 0);
  int rc = project_v2m(ctx, ctx->com_before, ctx->modes_before, st);
  if (rc) return rc;
  rc = project_v2m(ctx, ctx->err_v, ctx->modes_res, st);
  if (rc) return rc;
  dim3 grid((c.state_modes + 127) / 128, c.n_env);
  build_state_kernel<<<grid, 128, 0, st>>>(ctx->state, ctx->ldst, ctx->hist, c.n_hist, ctx->hist_head, ctx->modes_before,
                                           ctx->modes_res, ctx->ldm, (const int*)ctx->tab[AOM_T_STATE_MAP][0], c.state_modes,
                                           (const float*)ctx->tab[AOM_T_NORM_DM_MEAN][0], (const float*)ctx->tab[AOM_T_NORM_DM_STD][0],
                                           (const float*)ctx->tab[AOM_T_NORM_RES_MEAN][0], (const float*)ctx->tab[AOM_T_NORM_RES_STD][0],
                                           c.n_env);
  KCHECK();
  if (c.n_hist > 0) ctx->hist_head = (ctx->hist_head + 1) % c.n_hist;
  return end_first_steps(ctx, st);
}

extern "C" int aom_reward(aom_ctx* ctx, float factor, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  const aom_config& c = ctx->cfg;
  if (!ctx->reward) return fail(ctx, AOM_ERR_STATE, "n_agents is 0 in this configuration");
  NEED(AOM_T_AGENT_REWARD, 0);
  long long threads = (long long)c.n_env * c.n_agents * 32;
  reward_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctx->modes_res, ctx->ldm,
                                                                                     (const int*)ctx->tab[AOM_T_AGENT_REWARD][0],
                                                                                     c.n_agents, c.n_env, factor, ctx->reward);
  KCHECK();
  return AOM_OK;
}

extern "C" int aom_actor_forward(aom_ctx* ctx, int eval_mode, void* stream) {
  if (!ctx) return AOM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const aom_config& c = ctx->cfg;
  if (c.n_agents <= 0 || !ctx->state) return fail(ctx, AOM_ERR_STATE, "no agents / state configured");
  NEED(AOM_T_AGENT_IDX, 0); NEED(AOM_T_AGENT_ACT, 0); NEED(AOM_T_ACTOR_W1, 0); NEED(AOM_T_ACTOR_B1, 0);
  NEED(AOM_T_ACTOR_W2, 0); NEED(AOM_T_ACTOR_B2, 0); NEED(AOM_T_ACTOR_WH, 0); NEED(AOM_T_ACTOR_BH, 0);
  const int E = c.n_env, A = c.n_agents;
  actor_gather_kernel<<<E, 256, 0, st>>>(ctx->state, ctx->ldst, (const int*)ctx->tab[AOM_T_AGENT_IDX][0], c.actor_in,
                                         ctx->ld_ain, E, A, ctx->aX);
  KCHECK();
  int rc = launch_gemm(ctx, 0, ctx->aX, ctx->ld_ain, (long long)E * ctx->ld_ain, (const float*)ctx->tab[AOM_T_ACTOR_W1][0],
                       ctx->ld_ain, (long long)c.actor_hidden * ctx->ld_ain, ctx->aH1, ctx->ld_ah, (long long)E * ctx->ld_ah, E,
                       c.actor_hidden, c.actor_in, (const float*)ctx->tab[AOM_T_ACTOR_B1][0], c.actor_hidden, 1, A, st, nullptr, 0, false,
                       ctx->actor_bt[0], (long long)ctx->actor_bt_per[0]);
  if (rc) return rc;
  rc = launch_gemm(ctx, 0, ctx->aH1, ctx->ld_ah, (long long)E * ctx->ld_ah, (const float*)ctx->tab[AOM_T_ACTOR_W2][0], ctx->ld_ah,
                   (long long)c.actor_hidden * ctx->ld_ah, ctx->aH2, ctx->ld_ah, (long long)E * ctx->ld_ah, E, c.actor_hidden,
                   c.actor_hidden, (const float*)ctx->tab[AOM_T_ACTOR_B2][0], c.actor_hidden, 1, A, st, nullptr, 0, false,
                   ctx->actor_bt[1], (long long)ctx->actor_bt_per[1]);
  if (rc) return rc;
  rc = launch_gemm(ctx, 0, ctx->aH2, ctx->ld_ah, (long long)E * ctx->ld_ah, (const float*)ctx->tab[AOM_T_ACTOR_WH][0], ctx->ld_ah,
                   (long long)2 * c.actor_out * ctx->ld_ah, ctx->aHO, ctx->ld_aho, (long long)E * ctx->ld_aho, E, 2 * c.actor_out,
                   c.actor_hidden, (const float*)ctx->tab[AOM_T_ACTOR_BH][0], 2 * c.actor_out, 0, A, st, nullptr, 0, false,
                   ctx->actor_bt[2], (long long)ctx->actor_bt_per[2]);
  if (rc) return rc;
  actor_sample_kernel<<<E, 256, 0, st>>>(ctx->aHO, ctx->ld_aho, c.actor_out, (const int*)ctx->tab[AOM_T_AGENT_ACT][0], E, A,
                                         c.log_sig_min, c.log_sig_max, c.pol_act_scale, c.pol_act_bias, eval_mode, ctx->step,
                                         ctx->k0, ctx->k1, ctx->action, ctx->action_mean, ctx->ldact,
                                         ctx->staggered ? ctx->step_env : nullptr, ctx->first);
  KCHECK();
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
  if (ctx->reward) { rc = aom_reward(ctx, ctx->cfg.reward_factor, stream); if (rc) return rc; }
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
  rc = aom_comp_wfs_image(ctx, keep ? 7 : 3, ctx->noise_env ? 0.f : ctx->noise_c, stream); if (rc) return rc;
  if (denoise) { rc = aom_denoise(ctx, nullptr, nullptr, 0, stream); if (rc) return rc; }
  rc = aom_do_centroids(ctx, stream); if (rc) return rc;
  rc = aom_do_control(ctx, stream); if (rc) return rc;
  if (ctx->state) { rc = aom_state_end(ctx, stream); if (rc) return rc; }
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
