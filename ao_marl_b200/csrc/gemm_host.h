// Host interface of the env-batched GEMMs (gemm.cu): C[b][m][n] = sum_k A[b][m][k] * B[b][n][k] (+ bias) (relu), or the
// integrator epilogue, on the tcgen05 kernel (gemm_tc.cuh) or the SIMT ones (gemm_kernels.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "../../include/aomarl.h"

struct GemmParams {
  const float* A; const float* B; float* C; const float* bias;
  int lda, ldb, ldc;
  int M, N, K;          // K valid columns; the launcher rounds it up to a multiple of 16 (operands are zero padded)
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

// The batched actor forward of all agents in one kernel (actor_fused_kernel, actor_tc.cuh): X[a][e][k] = state[e][idx[a][k]],
// H1 = relu(W1 X + b1), H2 = relu(W2 H1 + b2), heads = WH H2 + bh, then the tanh-Gaussian actions of actor_sample_kernel.
struct ActorParams {
  const float* state; int ldst, E;
  const int* idx; int actor_in;           // [A][actor_in] state column of each input, -1: none
  int hidden, heads, ldh;                 // hidden units, 2 actor_out head columns and their leading dimension
  int nkb_in, nkb_h;                      // k blocks of 16 of layer 1 (AOM_LD(actor_in)) and of layers 2, 3 (AOM_LD(hidden))
  int nt_hidden, nt_heads;                // 128-column tiles of the hidden and the head layers
  const float* w[3]; long long w_per[3];  // pre-tiled hi / lo weights (gtc_pretile_host) and their floats per agent
  const float* bias[3];                   // [A][hidden], [A][hidden], [A][heads]
  int actor_out; const int* act_slot;     // [A][actor_out] action column, -1: unmapped
  float log_sig_min, log_sig_max, act_scale, act_bias;
  int eval_mode; uint32_t step;
  const uint32_t *k0, *k1, *step_env;     // [E] Philox keys; per-environment decision counters or null (`step` for all)
  float *action, *action_mean; int lda;
};

// The per-environment form (aom_set_controller_env): CTA (t, a) runs agent a of policy slot tile_slot[t] on the
// environments tile_env[t][0..128) (-1: padding; ctrl_tiles_host.h).  Slot s's pre-tiled weights are ws[s][l], its biases
// bs[s][l], both laid out per agent as w / bias of the uniform form.
struct ActorEnvParams : ActorParams {
  const int *tile_slot, *tile_env;
  const float* ws[AOM_MAX_POLICIES][3];
  const float* bs[AOM_MAX_POLICIES][3];
};
template <bool PE>
using ActorArgs = std::conditional_t<PE, ActorEnvParams, ActorParams>;

// Whether actor_fused_kernel serves these shapes: hidden and head layers of at most two 128-column tiles, and the input
// row within the shared memory next to the stages.
bool actor_fused_fits(int actor_in, int hidden, int heads);
// Launches actor_fused_kernel over all agents on st; the caller checks the launch (cudaGetLastError).
void actor_fused_launch(const ActorParams& p, int n_agents, int* err_word, cudaStream_t st);
// The same over the n_tiles tiles of the per-environment form.
void actor_fused_env_launch(const ActorEnvParams& p, int n_tiles, int n_agents, int* err_word, cudaStream_t st);

// Sets the dynamic shared-memory size of every tcgen05 GEMM instantiation; once per context, before any launch.
cudaError_t gemm_init();

// Launches one GEMM of `batch` products with epilogue epi (0 plain, 1 integrator, 2 integrator with p.gain_env) on st.
// `exact`: float32 FFMA accumulation with round-to-nearest, else the tcgen05 kernel unless gemm_path is AOM_GEMM_SIMT,
// whose bounded waits raise the device error word err_word.  Returns AOM_OK, or an error code with its message in err;
// the caller checks the launch itself (cudaGetLastError).
int gemm_launch(GemmParams p, int epi, int batch, bool exact, int gemm_path, int num_sms, int* err_word, cudaStream_t st,
                char (&err)[512]);
