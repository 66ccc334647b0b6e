// Small per-environment vector kernels around the GEMMs: delay line, modal action injection,
// state assembly with history ring, per-agent reward, actor input gather and action sampling.
// Reference call sites are cited per kernel (paths relative to the reference root).
#pragma once
#include <cuda_runtime.h>
#include "rng.cuh"

// RtcCompass.apply_control -> sutra comp_voltage (rtcCompass.py:573-582): volt = com (delay 0) or the
// command stored at the previous call (delay 1); then the delay line shifts.
__global__ void apply_control_kernel(const float* com, float* com1, float* volts, int ld, size_t total,
                                     int delay, int comp_voltage) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  if (!comp_voltage) return;          // "directly apply the current voltage vector": volts unchanged
  float c = com[i];
  volts[i] = delay ? com1[i] : c;
  com1[i] = c;
}

// RlSupervisor.correction_modal_basis step 2 (rlSupervisor.py:799-813):
// modes[action_map[i]] += (a[i] * act_scale + act_bias) * freedom[action_map[i]]
// first [E] (or null): environments restarted by aom_reset_envs whose first step is pending take no action.
__global__ void inject_action_kernel(float* modes, int ldm, const float* action, int lda, const int* action_map,
                                     const float* freedom, int action_dim, int E, float act_scale, float act_bias,
                                     const int* first) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int e = blockIdx.y;
  if (i >= action_dim || e >= E) return;
  if (first && first[e]) return;
  int m = action_map[i];
  float a = action[(size_t)e * lda + i] * act_scale + act_bias;
  modes[(size_t)e * ldm + m] += a * freedom[m];
}

// AoEnv.linear_step state assembly (ao_env.py:871-909, 470-480, 507-561).  State blocks, in order:
// dm_history_{n_hist} (oldest) ... dm_history_1, dm_before_linear, dm_residual ; each (x - mean) / std.
// hist is a ring of n_hist un-normalised "before" vectors; `head` is the slot holding the oldest.
__global__ void build_state_kernel(float* state, int lds, float* hist, int n_hist, int head,
                                   const float* modes_before, const float* modes_res, int ldm,
                                   const int* state_map, int sm, const float* dm_mean, const float* dm_std,
                                   const float* res_mean, const float* res_std, int E) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  int e = blockIdx.y;
  if (j >= sm || e >= E) return;
  int m = state_map[j];
  float* st = state + (size_t)e * lds;
  float mean = dm_mean[j], sd = dm_std[j];
  for (int h = 0; h < n_hist; ++h) {
    int slot = (head + h) % n_hist;
    float v = hist[((size_t)slot * E + e) * sm + j];
    st[h * sm + j] = (v - mean) / sd;
  }
  float before = modes_before[(size_t)e * ldm + m];
  st[n_hist * sm + j] = (before - mean) / sd;
  float res = modes_res[(size_t)e * ldm + m];
  st[(n_hist + 1) * sm + j] = (res - res_mean[j]) / res_std[j];
  if (n_hist > 0) hist[((size_t)head * E + e) * sm + j] = before;   // overwrite the oldest slot
}

// TrainerRPC.divide_rewards_for_agents + get_separated_rewards (train_rpc.py:402-416, helper_rewards.py:14-22)
// one warp per (env, agent)
__global__ void reward_kernel(const float* modes_res, int ldm, const int* ranges, int n_agents, int E,
                              float factor, float* reward) {
  int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= E * n_agents) return;
  int e = w / n_agents, a = w % n_agents;
  int a0 = ranges[2 * a], a1 = ranges[2 * a + 1];
  const float* r = modes_res + (size_t)e * ldm;
  float s = 0.f;
  for (int m = a0 + lane; m < a1; m += 32) s = fmaf(r[m], r[m], s);
#pragma unroll
  for (int sft = 16; sft > 0; sft >>= 1) s += __shfl_xor_sync(0xffffffffu, s, sft);
  if (lane == 0) reward[(size_t)e * n_agents + a] = -factor * s / (float)(a1 - a0);
}

// TrainerRPC.divide_states_for_agents (train_rpc.py:418-427): X[a][e][i] = state[e][idx[a][i]]
// grid: E blocks of 256 threads; one block serves all agents of its environment (the state row stays in L1, the
// per-agent rows are written as contiguous runs) -- half a million 128-thread blocks were block-latency bound.
__global__ void __launch_bounds__(256) actor_gather_kernel(const float* __restrict__ state, int lds,
                                                           const int* __restrict__ idx, int actor_in, int ldx, int E,
                                                           int n_agents, float* __restrict__ X) {
  const int e = blockIdx.x;
  const float* srow = state + (size_t)e * lds;
  const int total = n_agents * ldx;
  for (int t = threadIdx.x; t < total; t += blockDim.x) {
    const int a = t / ldx, i = t - a * ldx;
    float v = 0.f;
    if (i < actor_in) {
      const int s = __ldg(idx + (size_t)a * actor_in + i);
      if (s >= 0) v = srow[s];
    }
    X[((size_t)a * E + e) * ldx + i] = v;
  }
}

// GaussianPolicy.sample(only_choosing_action=True) + TrainerRPC.report_action
// (model_rpc.py:131-144, train_rpc.py:667-675).  heads[a][e][0:out] = mean, [out:2 out] = log std.
// grid: E blocks of 256 threads, every block loops over (agent, output).
// step_env [E] (or null: `step` for every environment): each environment's own decision counter, advanced here except
// for an environment whose first step after aom_reset_envs is pending (first[e]): that step's action is not used.
__global__ void __launch_bounds__(256) actor_sample_kernel(const float* __restrict__ heads, int ldh, int actor_out,
                                                           const int* __restrict__ act_slot, int E, int n_agents,
                                                           float log_sig_min, float log_sig_max, float act_scale,
                                                           float act_bias, int eval_mode, uint32_t step,
                                                           const uint32_t* k0, const uint32_t* k1, float* action,
                                                           float* action_mean, int lda, uint32_t* step_env,
                                                           const int* first) {
  const int e = blockIdx.x;
  const uint32_t key0 = k0[e], key1 = k1[e];
  if (step_env) step = step_env[e];
  const int total = n_agents * actor_out;
  for (int t = threadIdx.x; t < total; t += blockDim.x) {
    const int a = t / actor_out, j = t - a * actor_out;
    const int slot = __ldg(act_slot + (size_t)a * actor_out + j);
    if (slot < 0) continue;
    const float* h = heads + ((size_t)a * E + e) * ldh;
    const float mu = h[j];
    const float ls = fminf(fmaxf(h[actor_out + j], log_sig_min), log_sig_max);
    const aom_u4 w = aom_philox((uint32_t)(j >> 2), step, AOM_TAG_ACTOR, (uint32_t)a, key0, key1);
    const float eps = aom_normal_of_block(w, j & 3);
    const float act = tanhf(mu + expf(ls) * eps) * act_scale + act_bias;
    const float mean = tanhf(mu) * act_scale + act_bias;
    action[(size_t)e * lda + slot] = eval_mode ? mean : act;
    action_mean[(size_t)e * lda + slot] = mean;
  }
  if (step_env) {
    __syncthreads();                                  // every thread has read the counter
    if (threadIdx.x == 0 && !first[e]) step_env[e] = step + 1;
  }
}

__global__ void pixel_noise_kernel(const float* lam, float* out, long long n, float noise, uint32_t k0,
                                   uint32_t k1, uint32_t frame, uint32_t wfs) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = aom_pixel_noise(lam[i], noise, (uint32_t)i, frame, wfs, k0, k1);
}

__global__ void copy_rows_kernel(const float* src, int lds_, float* dst, int ldd, int n, int E) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int e = blockIdx.y;
  if (i >= ldd || e >= E) return;
  dst[(size_t)e * ldd + i] = (i < n) ? src[(size_t)e * lds_ + i] : 0.f;
}

// ---------------------------------------------------------------------------------------------
// aom_reset_envs: restart listed environments while the others run on.
#define RESET_MAX_BUFS (17 + 4 * AOM_MAX_LAYERS)    // controller, state and Strehl rows + screen and ring state per layer
struct ResetEnvsParams {
  // per-environment buffers whose rows are zeroed: word (s * slot_stride + e * ld + i), s < slots, i < ld
  uint32_t* buf[RESET_MAX_BUFS];
  long long ld[RESET_MAX_BUFS], slot_stride[RESET_MAX_BUFS];
  int slots[RESET_MAX_BUFS];
  int nbuf;
  const int* envs;              // [K] environments to restart
  const uint32_t* seeds;        // [2][K] low, high words of their new seeds
  int K, E;
  uint32_t *k0, *k1;            // [E] Philox keys
  uint32_t* frame0;             // [E] noise frame of the environment's first sensor frame
  uint32_t* step_env;           // [E] actor decision counters
  int* le_n;                    // [2][E] long-exposure counts (main target, geometric target)
  int* first;                   // [E] first step pending
  uint32_t frame;
};

// grid (K, nbuf + 1): block (k, b < nbuf) zeroes the rows of buffer b of environment envs[k]; block (k, nbuf) sets its
// keys and counters.
__global__ void __launch_bounds__(256) reset_envs_kernel(const __grid_constant__ ResetEnvsParams P) {
  const int k = blockIdx.x, b = blockIdx.y, e = P.envs[k];
  if (b < P.nbuf) {
    uint32_t* base = P.buf[b] + (size_t)e * P.ld[b];
    for (int s = 0; s < P.slots[b]; ++s)
      for (long long i = threadIdx.x; i < P.ld[b]; i += blockDim.x) base[s * P.slot_stride[b] + i] = 0u;
    return;
  }
  if (threadIdx.x == 0) {
    P.k0[e] = P.seeds[k];
    P.k1[e] = P.seeds[P.K + k];
    P.frame0[e] = P.frame;
    P.step_env[e] = 0u;
    P.le_n[e] = 0;
    P.le_n[P.E + e] = 0;
    P.first[e] = 1;
  }
}

// The per-environment counters when the batch stops running in lockstep: every environment at the batch's counts.
__global__ void stagger_counters_kernel(uint32_t* frame0, uint32_t* step_env, int* le_n, int* first, int E, uint32_t step,
                                        int n_main, int n_geo) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  frame0[e] = 0u;
  step_env[e] = step;
  le_n[e] = n_main;
  le_n[E + e] = n_geo;
  first[e] = 0;
}
