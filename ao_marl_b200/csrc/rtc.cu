// Host side of the controller: the integrator and the modal projections (extrude_i8.cuh, or the GEMMs of gemm.cu), the
// RL vectors around them (rtc_kernels.cuh), the actor forward (actor_tc.cuh, or gather, three GEMMs and sampling for
// wide actors) and the per-environment controllers.  The gain, delay, keys and tables stay the context's and are read
// through RtcLinks.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "rtc_host.h"
#include "rtc_kernels.cuh"
#include "ctrl_tiles_host.h"
#include "dalloc.h"
#include "extrude_i8_host.h"
#include "gemm_host.h"
#include "gemm_tc_host.h"

static_assert(AOM_MAX_POLICIES <= AOM_MAX_LAYERS, "the actor tables of every policy slot live in tab[table][slot]");

enum { OP_CMAT, OP_V2M, OP_M2V };

struct Rtc {
  aom_config cfg;
  RtcLinks in;
  // the integer contraction (extrude_i8.cuh) of the operator products: digit planes of cmat, v2m, m2v (OP_*), and the
  // scratch of the main stream (the extrusion has its own on the side stream)
  OzOperator op[3];
  OzScratch oz;
  // actor weights of every policy slot as pre-split TF32 hi / lo planes in the tile order of gemm_tc_kernel (W1, W2, WH),
  // floats per agent
  float* actor_bt[AOM_MAX_POLICIES][3];
  size_t actor_bt_per[3];
  // per-environment controllers (rtc_set_controller), all null while every environment is on slot 0: the assignment
  // (host and device [E]), the tile list of the per-environment actor kernel (ctrl_tiles_host.h), the environments on
  // the integrator, the skip mask of ctrl_skip_kernel and the com rows rtc_rl_control keeps for them
  int32_t* ctrl_host;
  int *ctrl_dev, *ctrl_tile_slot, *ctrl_tile_env, *ctrl_integ, *ctrl_skip;
  float* ctrl_com;
  int ctrl_ntiles, ctrl_ninteg;
  float *err_v, *com, *com1, *com2, *volts, *com_before;
  float *modes, *modes_before, *modes_res, *state, *hist, *reward, *action, *action_mean;
  int lda, ldm, ldst, ldact, hist_head;
  float *aX, *aH1, *aH2, *aHO;   // the wide actors' inputs, hidden layers and heads [A][E][ld]
  int ld_ain, ld_ah, ld_aho;
  int closed;
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
    ++*r->in.launches;                                                                            \
    cudaError_t _e = cudaGetLastError();                                                          \
    if (_e != cudaSuccess)                                                                        \
      return report(err, AOM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define NEED(t, i)                                                                     \
  do {                                                                                 \
    if (!r->in.tab[t][i]) return report(err, AOM_ERR_STATE, "table %s[%d] not uploaded", #t, i); \
  } while (0)

template <typename T>
static const T* tab(const Rtc* r, int t, int i = 0) { return (const T*)r->in.tab[t][i]; }

int rtc_create(const aom_config& c, const RtcLinks& links, Rtc** out, char (&err)[512]) {
  Rtc* r = (Rtc*)calloc(1, sizeof(Rtc));
  *out = r;
  if (!r) return report(err, AOM_ERR_INVALID, "out of host memory");
  r->cfg = c;
  r->in = links;
  r->closed = 1;
  const size_t E = c.n_env;
  r->lda = AOM_LD(c.nactu);
  r->ldm = AOM_LD(c.nmodes > 0 ? c.nmodes : 1);
  float** rows[] = {&r->err_v, &r->com, &r->com1, &r->com2, &r->volts, &r->com_before};
  for (float** b : rows) CU(dalloc(b, E * r->lda));
  for (float** b : {&r->modes, &r->modes_before, &r->modes_res})
    if (c.nmodes > 0) CU(dalloc(b, E * r->ldm));
  if (c.state_dim > 0) {
    r->ldst = AOM_LD(c.state_dim);
    CU(dalloc(&r->state, E * r->ldst));
    if (c.n_hist > 0) CU(dalloc(&r->hist, (size_t)c.n_hist * E * c.state_modes));
  }
  if (c.action_dim > 0) {
    r->ldact = AOM_LD(c.action_dim);
    CU(dalloc(&r->action, E * r->ldact));
    CU(dalloc(&r->action_mean, E * r->ldact));
  }
  if (c.n_agents > 0) {
    CU(dalloc(&r->reward, E * c.n_agents));
    r->ld_ain = AOM_LD(c.actor_in);
    r->ld_ah = AOM_LD(c.actor_hidden);
    r->ld_aho = AOM_LD(2 * c.actor_out);
    const size_t A = c.n_agents;
    CU(dalloc(&r->aX, A * E * r->ld_ain));
    CU(dalloc(&r->aH1, A * E * r->ld_ah));
    CU(dalloc(&r->aH2, A * E * r->ld_ah));
    CU(dalloc(&r->aHO, A * E * r->ld_aho));
  }
  return AOM_OK;
}

static void ctrl_free(Rtc* r) {
  int** dev[] = {&r->ctrl_dev, &r->ctrl_tile_slot, &r->ctrl_tile_env, &r->ctrl_integ, &r->ctrl_skip};
  for (int** b : dev) { cudaFree(*b); *b = nullptr; }
  cudaFree(r->ctrl_com); r->ctrl_com = nullptr;
  free(r->ctrl_host); r->ctrl_host = nullptr;
  r->ctrl_ntiles = r->ctrl_ninteg = 0;
}

void rtc_destroy(Rtc* r) {
  if (!r) return;
  void* bufs[] = {r->err_v, r->com, r->com1, r->com2, r->volts, r->com_before, r->modes, r->modes_before, r->modes_res, r->state,
                  r->hist, r->reward, r->action, r->action_mean, r->aX, r->aH1, r->aH2, r->aHO};
  for (void* b : bufs) cudaFree(b);
  for (OzOperator& o : r->op) oz_operator_free(o);
  oz_scratch_free(r->oz);
  for (int s = 0; s < AOM_MAX_POLICIES; ++s)
    for (int i = 0; i < 3; ++i) cudaFree(r->actor_bt[s][i]);
  ctrl_free(r);
  free(r);
}

RtcView rtc_view(const Rtc* r) {
  return RtcView{r->err_v, r->com, r->com1, r->com2, r->volts, r->com_before, r->modes, r->modes_res, r->state, r->hist,
                 r->reward, r->action, r->action_mean, r->lda, r->ldm, r->ldst, r->ldact, r->hist_head};
}

// Operator o (OP_*): its table, the K columns of its input rows and the N of its output rows, and their leading dimensions
struct Op {
  int table, K, N, ldx, ldo;
};

static Op op_of(const Rtc* r, int o) {
  const aom_config& c = r->cfg;
  const Op ops[3] = {{AOM_T_CMAT, c.nslopes, c.nactu, AOM_LD(c.nslopes), r->lda},
                     {AOM_T_V2M, c.nactu, c.nmodes, r->lda, r->ldm},
                     {AOM_T_M2V, c.nmodes, c.nactu, r->ldm, r->lda}};
  return ops[o];
}

int rtc_set_table(Rtc* r, int table, int index, const void* host, char (&err)[512]) {
  const aom_config& c = r->cfg;
  for (int o = 0; o < 3; ++o) {
    const Op q = op_of(r, o);
    if (q.table == table) return oz_operator_upload(r->op[o], (const float*)host, q.N, AOM_LD(q.K), q.K, err);
  }
  if (table != AOM_T_ACTOR_W1 && table != AOM_T_ACTOR_W2 && table != AOM_T_ACTOR_WH) return AOM_OK;
  // the same weights pre-split into TF32 hi / lo planes in the tile order of gemm_tc_kernel: the actor GEMMs then take
  // their B operand by one bulk copy per stage instead of global loads + split + st.shared in the loader warps.  One
  // copy per policy slot (index)
  const int i = table == AOM_T_ACTOR_W1 ? 0 : table == AOM_T_ACTOR_W2 ? 1 : 2;
  const int K = i == 0 ? c.actor_in : c.actor_hidden, ldb = AOM_LD(K);
  const int rows = i == 2 ? 2 * c.actor_out : c.actor_hidden;
  const int ldc = AOM_LD(rows);                                   // the output's leading dimension fixes the n tiles
  const size_t per = gtc_pretile_floats(ldc, AOM_LD(K));
  float* h = (float*)calloc(per * (size_t)c.n_agents, sizeof(float));
  if (!h) return report(err, AOM_ERR_INVALID, "out of host memory");
  gtc_pretile_host((const float*)host, c.n_agents, (long long)rows * ldb, ldb, rows, ldc, AOM_LD(K), h);
  float*& bt = r->actor_bt[index][i];
  cudaFree(bt); bt = nullptr;
  cudaError_t e = cudaMalloc((void**)&bt, per * c.n_agents * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(bt, h, per * c.n_agents * sizeof(float), cudaMemcpyHostToDevice);
  free(h);
  if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "pre-tiled actor weights: %s", cudaGetErrorString(e));
  r->actor_bt_per[i] = per;
  return AOM_OK;
}

int rtc_clear(Rtc* r, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  const size_t E = c.n_env;
  float* rows[] = {r->err_v, r->com, r->com1, r->com2, r->volts, r->com_before};
  for (float* b : rows) CU(cudaMemsetAsync(b, 0, E * r->lda * 4, st));
  if (r->modes_res) CU(cudaMemsetAsync(r->modes_res, 0, E * r->ldm * 4, st));
  if (r->hist) CU(cudaMemsetAsync(r->hist, 0, (size_t)c.n_hist * E * c.state_modes * 4, st));
  if (r->state) CU(cudaMemsetAsync(r->state, 0, E * r->ldst * 4, st));
  if (r->action) CU(cudaMemsetAsync(r->action, 0, E * r->ldact * 4, st));
  r->hist_head = 0;
  return AOM_OK;
}

void rtc_set_loop(Rtc* r, int closed) { r->closed = closed ? 1 : 0; }

// ---------------------------------------------------------------------------------------------
// per-environment controllers

// Whether policy slot s has its six actor tables (and the pre-split copies of its weights)
static bool slot_ready(const Rtc* r, int s) {
  for (int t = AOM_T_ACTOR_W1; t <= AOM_T_ACTOR_BH; ++t)
    if (!r->in.tab[t][s]) return false;
  return r->actor_bt[s][0] && r->actor_bt[s][1] && r->actor_bt[s][2];
}

int rtc_set_controller(Rtc* r, const int32_t* ctrl, char (&err)[512]) {
  const int E = r->cfg.n_env;
  bool uniform = true;
  for (int e = 0; ctrl && e < E; ++e) {
    const int v = ctrl[e];
    if (v < AOM_CTRL_INTEGRATOR || v >= AOM_MAX_POLICIES)
      return report(err, AOM_ERR_INVALID, "aom_set_controller_env: environment %d: controller %d is neither a policy slot in "
                    "[0, %d) nor AOM_CTRL_INTEGRATOR", e, v, AOM_MAX_POLICIES);
    if (v >= 0 && !slot_ready(r, v))
      return report(err, AOM_ERR_STATE, "aom_set_controller_env: environment %d: policy slot %d does not have its six actor "
                    "tables (AOM_T_ACTOR_W1 .. AOM_T_ACTOR_BH at index %d)", e, v, v);
    uniform = uniform && v == 0;
  }
  CU(cudaDeviceSynchronize());                       // a kernel in flight may still read the old tile list
  ctrl_free(r);
  if (uniform) return AOM_OK;
  const int tmax = ctl_tiles_max(E);
  int32_t* ts = (int32_t*)malloc((size_t)tmax * (1 + CTL_TILE) * sizeof(int32_t));
  int32_t* integ = (int32_t*)malloc((size_t)E * sizeof(int32_t));
  r->ctrl_host = (int32_t*)malloc((size_t)E * sizeof(int32_t));
  if (!ts || !integ || !r->ctrl_host) {
    free(ts); free(integ); ctrl_free(r);
    return report(err, AOM_ERR_INVALID, "out of host memory");
  }
  memcpy(r->ctrl_host, ctrl, (size_t)E * sizeof(int32_t));
  int32_t* te = ts + tmax;
  const int nt = ctl_build_tiles(ctrl, E, ts, te, integ, &r->ctrl_ninteg);
  r->ctrl_ntiles = nt;
  cudaError_t ce = dalloc(&r->ctrl_dev, (size_t)E);
  if (ce == cudaSuccess) ce = dalloc(&r->ctrl_tile_slot, (size_t)tmax);
  if (ce == cudaSuccess) ce = dalloc(&r->ctrl_tile_env, (size_t)tmax * CTL_TILE);
  if (ce == cudaSuccess) ce = dalloc(&r->ctrl_integ, (size_t)E);
  if (ce == cudaSuccess) ce = dalloc(&r->ctrl_skip, (size_t)E);
  if (ce == cudaSuccess && r->ctrl_ninteg) ce = dalloc(&r->ctrl_com, (size_t)r->ctrl_ninteg * r->lda);
  if (ce == cudaSuccess) ce = cudaMemcpy(r->ctrl_dev, ctrl, (size_t)E * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess && nt) ce = cudaMemcpy(r->ctrl_tile_slot, ts, (size_t)nt * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess && nt)
    ce = cudaMemcpy(r->ctrl_tile_env, te, (size_t)nt * CTL_TILE * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess && r->ctrl_ninteg)
    ce = cudaMemcpy(r->ctrl_integ, integ, (size_t)r->ctrl_ninteg * sizeof(int32_t), cudaMemcpyHostToDevice);
  free(ts); free(integ);
  if (ce != cudaSuccess) {
    ctrl_free(r);
    return report(err, AOM_ERR_CUDA, "aom_set_controller_env: %s (the batch is back on slot 0)", cudaGetErrorString(ce));
  }
  return AOM_OK;
}

void rtc_get_controller(const Rtc* r, int32_t* ctrl, int* per_env) {
  if (per_env) *per_env = r->ctrl_host != nullptr;
  for (int e = 0; ctrl && e < r->cfg.n_env; ++e) ctrl[e] = r->ctrl_host ? r->ctrl_host[e] : 0;
}

bool rtc_integrators(const Rtc* r) { return r->ctrl_ninteg > 0; }

// The skip mask of the environments on the integrator and those whose first step is pending, when some environment is
// on the integrator; else the first-step flags (null when none is set)
static const int* ctrl_skip(Rtc* r, const RtcCounters& n, cudaStream_t st, int* rc, char (&err)[512]) {
  const int E = r->cfg.n_env;
  const int* first = n.first_any ? n.first : nullptr;
  *rc = AOM_OK;
  if (!r->ctrl_ninteg) return first;
  ctrl_skip_kernel<<<(E + 255) / 256, 256, 0, st>>>(r->ctrl_dev, first, r->ctrl_skip, E);
  ++*r->in.launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) *rc = report(err, AOM_ERR_CUDA, "ctrl_skip_kernel launch failed: %s", cudaGetErrorString(e));
  return r->ctrl_skip;
}

// com rows of the environments on the integrator around rtc_rl_control's two products (restore 0: save, 1: write back)
static int ctrl_com_rows(Rtc* r, int restore, cudaStream_t st, char (&err)[512]) {
  if (!r->ctrl_ninteg) return AOM_OK;
  env_rows_kernel<<<dim3((r->lda + 255) / 256, r->ctrl_ninteg), 256, 0, st>>>(r->com, r->ctrl_com, r->lda, r->ctrl_integ,
                                                                            r->ctrl_ninteg, restore);
  KCHECK();
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
// out[E][ldo] = X[E][ldx] . OP^T for operator o.  On the tcgen05 path, once the operator has its digit planes: the exact
// integer contraction with one rounding to float32 -- the oracle's float64 evaluation of the controller products
// (oracle/loop.py); else the GEMM.  integrator: the least-squares integrator epilogue, err = out = -product and
// com += gain * err while the loop is closed, with one gain per environment when the store has them.
static int product(Rtc* r, int o, const float* X, float* out, bool integrator, cudaStream_t st, char (&err)[512]) {
  const Op q = op_of(r, o);
  const int E = r->cfg.n_env;
  const EnvCond& gain = *r->in.gain;
  if (r->in.opt[AOM_OPT_GEMM_PATH] == AOM_GEMM_TCGEN05 && r->op[o].planes) {
    const OzOperator& P = r->op[o];
    const int MT = (E + OZ_BM - 1) / OZ_BM;
    CU(oz_scratch_reserve(r->oz, MT, P.kb, E, st));
    OzSliceParams sl;
    sl.X = X; sl.ld = q.ldx; sl.K = q.K; sl.E = E; sl.KB = P.kb; sl.Zs = r->oz.zs; sl.ev = r->oz.ev;
    OzGemmParams m;
    memset(&m, 0, sizeof(m));
    m.Zs = r->oz.zs; m.ABs = P.planes; m.ev = r->oz.ev; m.ea = P.ea; m.out = out; m.ldo = q.ldo;
    m.E = E; m.N = q.N; m.KB = P.kb; m.closed = r->closed; m.err = r->in.err_word; m.gain = gain.common;
    if (integrator) { m.com = r->com; m.ldcom = r->lda; m.gain_env = gain.dev; }
    cudaError_t le = oz_product_launch(sl, m, integrator, MT, P.nt, st);
    if (le != cudaSuccess) return report(err, AOM_ERR_CUDA, "oz_product_launch: %s", cudaGetErrorString(le));
    *r->in.launches += 2;
    return AOM_OK;
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.A = X; p.lda = q.ldx; p.B = tab<float>(r, q.table); p.ldb = q.ldx; p.C = out; p.ldc = q.ldo;
  p.M = E; p.N = q.N; p.K = q.K;
  if (integrator) { p.com = r->com; p.ldcom = r->lda; p.gain = gain.common; p.closed = r->closed; p.gain_env = gain.dev; }
  const int epi = !integrator ? 0 : gain.dev ? 2 : 1;
  int rc = gemm_launch(p, epi, 1, false, r->in.opt[AOM_OPT_GEMM_PATH], r->in.num_sms, r->in.err_word, st, err);
  if (rc) return rc;
  KCHECK();
  return AOM_OK;
}

int rtc_do_control(Rtc* r, const float* slopes, cudaStream_t st, char (&err)[512]) {
  NEED(AOM_T_CMAT, 0);
  return product(r, OP_CMAT, slopes, r->err_v, true, st, err);
}

int rtc_set_rows(Rtc* r, int buffer, const float* src, int ld, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  if (ld < c.nactu) return report(err, AOM_ERR_INVALID, "Dimension mismatch");
  dim3 grid((r->lda + 255) / 256, c.n_env);
  copy_rows_kernel<<<grid, 256, 0, st>>>(src, ld, buffer == AOM_B_COM ? r->com : r->volts, r->lda, c.nactu, c.n_env);
  KCHECK();
  return AOM_OK;
}

int rtc_apply_control(Rtc* r, int comp_voltage, cudaStream_t st, char (&err)[512]) {
  const size_t total = (size_t)r->cfg.n_env * r->lda;
  const EnvCond& delay = *r->in.delay;
  delay_line_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(r->com, r->com1, r->com2, r->volts, r->lda, total,
                                                                      delay.common, delay.dev, comp_voltage);
  KCHECK();
  return AOM_OK;
}

int rtc_reset_dm(Rtc* r, cudaStream_t st, char (&err)[512]) {
  CU(cudaMemsetAsync(r->volts, 0, (size_t)r->cfg.n_env * r->lda * 4, st));
  return AOM_OK;
}

// ---------------------------------------------------------------------------------------------
int rtc_rl_control(Rtc* r, const float* daction, const RtcCounters& n, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  NEED(AOM_T_M2V, 0); NEED(AOM_T_FREEDOM, 0); NEED(AOM_T_ACTION_MAP, 0);
  const float* act = daction ? daction : r->action;
  if (!act) return report(err, AOM_ERR_STATE, "no action buffer");
  NEED(AOM_T_V2M, 0);
  // environments on the integrator: m2v . v2m is not the identity, so their com rows are kept aside and written back
  int rc = ctrl_com_rows(r, 0, st, err);
  if (rc) return rc;
  const int* skip = ctrl_skip(r, n, st, &rc, err);
  if (rc) return rc;
  rc = product(r, OP_V2M, r->com, r->modes, false, st, err);
  if (rc) return rc;
  dim3 grid((c.action_dim + 127) / 128, c.n_env);
  inject_action_kernel<<<grid, 128, 0, st>>>(r->modes, r->ldm, act, r->ldact, tab<int>(r, AOM_T_ACTION_MAP),
                                             tab<float>(r, AOM_T_FREEDOM), c.action_dim, c.n_env, c.env_act_scale,
                                             c.env_act_bias, skip);
  KCHECK();
  rc = product(r, OP_M2V, r->modes, r->com, false, st, err);
  if (rc) return rc;
  return ctrl_com_rows(r, 1, st, err);
}

int rtc_state_begin(Rtc* r, cudaStream_t st, char (&err)[512]) {
  CU(cudaMemcpyAsync(r->com_before, r->com, (size_t)r->cfg.n_env * r->lda * 4, cudaMemcpyDeviceToDevice, st));
  return AOM_OK;
}

int rtc_state_end(Rtc* r, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  if (!r->state) return report(err, AOM_ERR_STATE, "state_dim is 0 in this configuration");
  NEED(AOM_T_STATE_MAP, 0); NEED(AOM_T_NORM_DM_MEAN, 0); NEED(AOM_T_NORM_DM_STD, 0);
  NEED(AOM_T_NORM_RES_MEAN, 0); NEED(AOM_T_NORM_RES_STD, 0); NEED(AOM_T_V2M, 0);
  int rc = product(r, OP_V2M, r->com_before, r->modes_before, false, st, err);
  if (rc) return rc;
  rc = product(r, OP_V2M, r->err_v, r->modes_res, false, st, err);
  if (rc) return rc;
  dim3 grid((c.state_modes + 127) / 128, c.n_env);
  build_state_kernel<<<grid, 128, 0, st>>>(r->state, r->ldst, r->hist, c.n_hist, r->hist_head, r->modes_before,
                                           r->modes_res, r->ldm, tab<int>(r, AOM_T_STATE_MAP), c.state_modes,
                                           tab<float>(r, AOM_T_NORM_DM_MEAN), tab<float>(r, AOM_T_NORM_DM_STD),
                                           tab<float>(r, AOM_T_NORM_RES_MEAN), tab<float>(r, AOM_T_NORM_RES_STD),
                                           c.n_env);
  KCHECK();
  if (c.n_hist > 0) r->hist_head = (r->hist_head + 1) % c.n_hist;
  return AOM_OK;
}

int rtc_reward(Rtc* r, float factor, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  if (!r->reward) return report(err, AOM_ERR_STATE, "n_agents is 0 in this configuration");
  NEED(AOM_T_AGENT_REWARD, 0);
  const long long threads = (long long)c.n_env * c.n_agents * 32;
  reward_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(r->modes_res, r->ldm, tab<int>(r, AOM_T_AGENT_REWARD),
                                                                   c.n_agents, c.n_env, factor, r->reward);
  KCHECK();
  return AOM_OK;
}

int rtc_actor_forward(Rtc* r, int eval_mode, const RtcCounters& n, cudaStream_t st, char (&err)[512]) {
  const aom_config& c = r->cfg;
  if (c.n_agents <= 0 || !r->state) return report(err, AOM_ERR_STATE, "no agents / state configured");
  NEED(AOM_T_AGENT_IDX, 0); NEED(AOM_T_AGENT_ACT, 0);
  const int E = c.n_env, A = c.n_agents;
  const int path = r->in.opt[AOM_OPT_GEMM_PATH];
  const bool fused = path != AOM_GEMM_SIMT && actor_fused_fits(c.actor_in, c.actor_hidden, 2 * c.actor_out);
  if (r->ctrl_host) {
    // per-environment controllers: the slots' tables were checked by rtc_set_controller
    if (!fused)
      return report(err, AOM_ERR_UNSUPPORTED, "per-environment controllers are implemented in the fused actor kernel only, "
                    "which does not serve %s", path == AOM_GEMM_SIMT ? "the SIMT GEMM path" :
                    "hidden or head layers wider than 256 columns");
  } else {
    NEED(AOM_T_ACTOR_W1, 0); NEED(AOM_T_ACTOR_B1, 0); NEED(AOM_T_ACTOR_W2, 0); NEED(AOM_T_ACTOR_B2, 0);
    NEED(AOM_T_ACTOR_WH, 0); NEED(AOM_T_ACTOR_BH, 0);
  }
  const int bias_t[3] = {AOM_T_ACTOR_B1, AOM_T_ACTOR_B2, AOM_T_ACTOR_BH};
  if (fused) {
    ActorEnvParams q;
    memset(&q, 0, sizeof(q));
    ActorParams& p = q;
    p.state = r->state; p.ldst = r->ldst; p.E = E;
    p.idx = tab<int>(r, AOM_T_AGENT_IDX); p.actor_in = c.actor_in;
    p.hidden = c.actor_hidden; p.heads = 2 * c.actor_out; p.ldh = r->ld_aho;
    p.nkb_in = r->ld_ain / 16; p.nkb_h = r->ld_ah / 16;
    p.nt_hidden = (r->ld_ah + 127) / 128; p.nt_heads = (r->ld_aho + 127) / 128;
    for (int i = 0; i < 3; ++i) {
      p.w[i] = r->actor_bt[0][i]; p.w_per[i] = (long long)r->actor_bt_per[i]; p.bias[i] = tab<float>(r, bias_t[i]);
    }
    p.actor_out = c.actor_out; p.act_slot = tab<int>(r, AOM_T_AGENT_ACT);
    p.log_sig_min = c.log_sig_min; p.log_sig_max = c.log_sig_max; p.act_scale = c.pol_act_scale; p.act_bias = c.pol_act_bias;
    p.eval_mode = eval_mode; p.step = n.step; p.k0 = r->in.k0; p.k1 = r->in.k1; p.step_env = n.step_env;
    p.action = r->action; p.action_mean = r->action_mean; p.lda = r->ldact;
    if (!r->ctrl_host) {
      actor_fused_launch(p, A, r->in.err_word, st);
      KCHECK();
    } else if (r->ctrl_ntiles) {
      q.tile_slot = r->ctrl_tile_slot; q.tile_env = r->ctrl_tile_env;
      for (int s = 0; s < AOM_MAX_POLICIES; ++s)
        for (int i = 0; i < 3; ++i) { q.ws[s][i] = r->actor_bt[s][i]; q.bs[s][i] = tab<float>(r, bias_t[i], s); }
      actor_fused_env_launch(q, r->ctrl_ntiles, A, r->in.err_word, st);
      KCHECK();
    }
    // the decision counters advance after every agent's CTAs have read them (not those of integrator environments)
    if (n.step_env) {
      int rc = AOM_OK;
      const int* skip = r->ctrl_ninteg ? ctrl_skip(r, n, st, &rc, err) : n.first;
      if (rc) return rc;
      step_env_advance_kernel<<<(E + 255) / 256, 256, 0, st>>>(n.step_env, skip, E);
      KCHECK();
    }
    return AOM_OK;
  }
  // hidden or head layers wider than two column tiles, or the SIMT path: gather, three GEMMs, sampling
  actor_gather_kernel<<<E, 256, 0, st>>>(r->state, r->ldst, tab<int>(r, AOM_T_AGENT_IDX), c.actor_in, r->ld_ain, E, A,
                                         r->aX);
  KCHECK();
  const struct {
    int w;
    const float* x;
    int ldx;
    float* y;
    int ldy, K, N, relu;
  } layer[3] = {{AOM_T_ACTOR_W1, r->aX, r->ld_ain, r->aH1, r->ld_ah, c.actor_in, c.actor_hidden, 1},
                {AOM_T_ACTOR_W2, r->aH1, r->ld_ah, r->aH2, r->ld_ah, c.actor_hidden, c.actor_hidden, 1},
                {AOM_T_ACTOR_WH, r->aH2, r->ld_ah, r->aHO, r->ld_aho, c.actor_hidden, 2 * c.actor_out, 0}};
  for (int i = 0; i < 3; ++i) {
    const auto& L = layer[i];
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.A = L.x; p.lda = L.ldx; p.sA = (long long)E * L.ldx;
    p.B = tab<float>(r, L.w); p.ldb = L.ldx; p.sB = (long long)L.N * L.ldx;
    p.C = L.y; p.ldc = L.ldy; p.sC = (long long)E * L.ldy;
    p.M = E; p.N = L.N; p.K = L.K;
    p.bias = tab<float>(r, bias_t[i]); p.sBias = L.N; p.relu = L.relu;
    p.Bt = r->actor_bt[0][i]; p.sBt = (long long)r->actor_bt_per[i];
    int rc = gemm_launch(p, 0, A, false, path, r->in.num_sms, r->in.err_word, st, err);
    if (rc) return rc;
    KCHECK();
  }
  actor_sample_kernel<<<E, 256, 0, st>>>(r->aHO, r->ld_aho, c.actor_out, tab<int>(r, AOM_T_AGENT_ACT), E, A,
                                         c.log_sig_min, c.log_sig_max, c.pol_act_scale, c.pol_act_bias, eval_mode, n.step,
                                         r->in.k0, r->in.k1, r->action, r->action_mean, r->ldact, n.step_env, n.first);
  KCHECK();
  return AOM_OK;
}
