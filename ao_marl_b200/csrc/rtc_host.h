// Host interface of the controller (rtc.cu): the integrator and the modal projections with the operator digit planes
// of their exact integer products, the RL vectors around them (action injection, state with its history ring, rewards),
// the actor forward of every policy slot with the slots' pre-split weights, and the per-environment controller
// assignment.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/aomarl.h"
#include "env_cond.h"

struct Rtc;

// What the controller reads from its context on every call; each pointer stays valid for the context's life.
struct RtcLinks {
  const EnvCond* gain;                     // the integrator gain of the conditions store
  const EnvCond* delay;                    // the controller delay (frames) of the conditions store
  void* const (*tab)[AOM_MAX_LAYERS];      // the device tables [aom_table][index]
  const int* opt;                          // the options [aom_option]: GEMM path
  const uint32_t* k0;                      // Philox keys [E]
  const uint32_t* k1;
  int* err_word;                           // device error word raised by bounded waits
  uint64_t* launches;                      // the context's count of kernel launches
  int num_sms;
};

// The context's counters a call reads: the batch's decision count; while the batch is staggered the per-environment
// decision counters (else null); the first-step flags (null until the batch was first staggered) and whether one may
// be set.
struct RtcCounters {
  uint32_t step;
  uint32_t* step_env;
  const int* first;
  bool first_any;
};

// The controller's device buffers, [E] rows each (hist: [n_hist][E][state_modes], slot hist_head the oldest; com1 /
// com2 the commands of the last two aom_apply_control calls before this one); null when the configuration has none.
struct RtcView {
  float *err, *com, *com1, *com2, *volts, *com_before;
  float *modes, *modes_res, *state, *hist, *reward, *action, *action_mean;
  int lda, ldm, ldst, ldact, hist_head;
};

// Every function returns AOM_OK, or an error code with its message in err.  *out is set even on failure, for
// rtc_destroy.
int rtc_create(const aom_config& c, const RtcLinks& links, Rtc** out, char (&err)[512]);
void rtc_destroy(Rtc* r);

RtcView rtc_view(const Rtc* r);

// Takes note of an uploaded table (aom_set_table), before the context keeps it: the digit planes of cmat / v2m / m2v,
// the pre-split planes of a policy slot's actor weights.  A non-finite operator is refused and changes nothing.
int rtc_set_table(Rtc* r, int table, int index, const void* host, char (&err)[512]);

// Zeroes the loop vectors and the history ring (aom_reset)
int rtc_clear(Rtc* r, cudaStream_t st, char (&err)[512]);
void rtc_set_loop(Rtc* r, int closed);

// The controller of every environment (aom_set_controller_env; null: slot 0 for all), and back
int rtc_set_controller(Rtc* r, const int32_t* ctrl, char (&err)[512]);
void rtc_get_controller(const Rtc* r, int32_t* ctrl, int* per_env);
// Whether some environment is on the integrator: the batch then needs per-environment counters
bool rtc_integrators(const Rtc* r);

// The integrator on the slopes [E][AOM_LD(nslopes)] (aom_do_control)
int rtc_do_control(Rtc* r, const float* slopes, cudaStream_t st, char (&err)[512]);
// Rows of com (buffer AOM_B_COM, aom_set_command) or volts (AOM_B_VOLTS, aom_set_dm_volts) from src [E][ld]
int rtc_set_rows(Rtc* r, int buffer, const float* src, int ld, cudaStream_t st, char (&err)[512]);
// The delay line with each environment's delay (the store's array, else its common value)
int rtc_apply_control(Rtc* r, int comp_voltage, cudaStream_t st, char (&err)[512]);
int rtc_reset_dm(Rtc* r, cudaStream_t st, char (&err)[512]);

// The half-steps of the RL loop (aom_rl_control, aom_state_begin, aom_state_end, aom_reward, aom_actor_forward)
int rtc_rl_control(Rtc* r, const float* daction, const RtcCounters& n, cudaStream_t st, char (&err)[512]);
int rtc_state_begin(Rtc* r, cudaStream_t st, char (&err)[512]);
int rtc_state_end(Rtc* r, cudaStream_t st, char (&err)[512]);
int rtc_reward(Rtc* r, float factor, cudaStream_t st, char (&err)[512]);
int rtc_actor_forward(Rtc* r, int eval_mode, const RtcCounters& n, cudaStream_t st, char (&err)[512]);
