/* aomarl.h -- C ABI of libaomarl.so: batched closed-loop adaptive-optics environment step on B200.
 *
 * The reference (Tomeu7/AO-MARL) has no C interface for this path: its Python supervisor calls the
 * un-vendored COMPASS pybind11 objects (shesha/sutra_wrap.py:46-72).  Every entry point below names
 * the reference call it replaces (paths relative to the reference root).  A maintainer binds these
 * with ctypes exactly as ao_marl_b200/lib.py does; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - one aom_ctx per GPU / process; it owns all persistent simulator state for E environments
 *   - every op is asynchronous on the cudaStream_t passed as `void* stream`
 *   - per-environment vectors are row-major [E][ld], ld = AOM_LD(n) floats, pad columns kept at 0
 *   - pupil-plane arrays are [y][x], x fastest (flat index x + n*y, as the reference's integer maps)
 *   - return value: 0 on success, negative aom_status otherwise; aom_last_error() gives the text
 */
#ifndef AOMARL_H
#define AOMARL_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AOM_MAX_LAYERS 8
#define AOM_WFS_TIMERS 64             /* sensor-kernel launches timed between two aom_wfs_time_ms calls */
#define AOM_LD(n) (((n) + 15) & ~15)

typedef struct aom_ctx aom_ctx;

typedef enum aom_status {
  AOM_OK = 0,
  AOM_ERR_INVALID = -1,     /* bad argument / dimension mismatch (reference: ValueError, rtcCompass.py:471-472) */
  AOM_ERR_CUDA = -2,        /* CUDA runtime error */
  AOM_ERR_UNSUPPORTED = -3, /* configuration outside the hot-path scope */
  AOM_ERR_STATE = -4        /* missing table / op called before its prerequisites */
} aom_status;

/* Scalar description of one configuration (filled from the host builders, ao_marl_b200/tables.py). */
typedef struct aom_config {
  int32_t n_env;                        /* E */
  int32_t n;                            /* mpupil side (p_geom._n, geom_init.py:833) */
  /* atmosphere (atmos_init.py:76-132) */
  int32_t n_layers;
  int32_t screen_dim[AOM_MAX_LAYERS];
  int32_t stencil_size[AOM_MAX_LAYERS];
  float deltax[AOM_MAX_LAYERS];         /* wind step, pixels / frame */
  float deltay[AOM_MAX_LAYERS];
  float amp[AOM_MAX_LAYERS];            /* innovation amplitude r0_px^(-5/6) * 0.5/(2 pi), microns */
  float wfs_xoff[AOM_MAX_LAYERS];       /* wfs_init.py:175-185 */
  float wfs_yoff[AOM_MAX_LAYERS];
  /* Shack-Hartmann sensor (geom_init.py:168-340, 622-811) */
  int32_t nxsub, nvalid, pdiam, npix, nfft, nrebin;
  float lambda_um;
  float nphotons;
  float noise;                          /* <0 none, 0 photon, >0 photon + read (e-) */
  float pixsize;                        /* arcsec / detector pixel (rtc_init.py:217) */
  float cog_offset;                     /* npix/2 - 0.5 (rtc_init.py:208) */
  int32_t wfs_index;                    /* RNG sub-stream */
  /* mirrors (dm_init.py:330-509, 661-694) */
  int32_t pzt_nact;
  int32_t stamp_size;                   /* influsize */
  int32_t pzt_off;                      /* (dim_dm - n)/2, wfs_init.py:196-204 */
  int32_t pzt_pitch;                    /* actuator pitch in pixels (integer on the production grids) */
  int32_t pzt_grid_n;                   /* side of the actuator lattice behind act_map */
  int32_t pzt_i1_0;                     /* i1 of lattice column 0 (DM-support pixels) */
  int32_t pzt_j1_0;
  int32_t tt_dim;
  int32_t tt_off;
  /* controller (rtc_init.py:451-513) */
  int32_t nactu, nslopes, nmodes;
  float gain;
  int32_t delay;                        /* 0 or 1 frames of command latency (p_controller.delay) */
  /* RL layer (ao_env.py, train_rpc.py) */
  int32_t n_hist;                       /* number_of_previous_dm */
  int32_t state_modes;                  /* modes kept per state block (all modes when windowed, else the action range) */
  int32_t state_dim;                    /* (n_hist + 2) * state_modes */
  float env_act_scale, env_act_bias;    /* normalization_{std,mean}_inside_environment (rlSupervisor.py:724-726) */
  float pol_act_scale, pol_act_bias;    /* gaussian_std / gaussian_mu of the policies (model_rpc.py:115-116) */
  float log_sig_min, log_sig_max;       /* -20 / LOG_SIG_MAX (model_rpc.py:12, 128) */
  int32_t n_agents;
  int32_t actor_in, actor_hidden, actor_out; /* padded common sizes of the batched actors */
  int32_t action_dim;                   /* length of the global action vector */
  float reward_factor;                  /* <factor> of reward_type "avg_squared_modes_<factor>" (helper_rewards.py:14-22,
                                           GlobalConfig.py:86); aom_step scales the per-agent rewards with it */
} aom_config;

/* Tables uploaded once after aom_create (host pointers; copied to the device). */
typedef enum aom_table {
  AOM_T_AB = 0,        /* float [N][ld(S+N)]   rows of A | B            index = layer   (iterkolmo.py:190-252) */
  AOM_T_STENCIL,       /* int32 [S]            +x stencil, flat x+N*y   index = layer   (iterkolmo.py:41-73)   */
  AOM_T_MPUPIL,        /* float [n][n]                                                (geom_init.py:845)     */
  AOM_T_HALFXY,        /* float [pdiam][pdiam]                                        (geom_init.py:690-701) */
  AOM_T_SUB_X0,        /* int32 [nvalid]       tile origin column in the mpupil frame (geom_init.py:673-685) */
  AOM_T_SUB_Y0,        /* int32 [nvalid]       tile origin row                                               */
  AOM_T_FLUX,          /* float [nvalid]       illuminated fraction, list order       (wfs_init.py:145)      */
  AOM_T_STAMP1D,       /* float [stamp_size]   separable factor of the actuator stamp (influ_util.py:139-183)*/
  AOM_T_ACT_MAP,       /* int32 [grid_n^2]     lattice cell -> actuator index or -1   (dm_init.py:414-427)   */
  AOM_T_TT_PLANES,     /* float [2][tt_dim][tt_dim]                                   (dm_init.py:661-694)   */
  AOM_T_CMAT,          /* float [nactu][ld(nslopes)]                                  (basis.py:229-256)     */
  AOM_T_V2M,           /* float [nmodes][ld(nactu)]   volts -> Btt modes (P)          (basis.py:362-443)     */
  AOM_T_M2V,           /* float [nactu][ld(nmodes)]   Btt modes -> volts (Btt)                               */
  AOM_T_FREEDOM,       /* float [nmodes]       action bound per mode                  (rlSupervisor.py:255-282)*/
  AOM_T_ACTION_MAP,    /* int32 [action_dim]   action element -> mode index           (rlSupervisor.py:677-691)*/
  AOM_T_STATE_MAP,     /* int32 [state_modes]  mode index of each state-block entry    (ao_env.py:482-505)     */
  AOM_T_NORM_DM_MEAN,  /* float [state_modes]  (ao_env.py:470-480, 279-301)                                  */
  AOM_T_NORM_DM_STD,
  AOM_T_NORM_RES_MEAN,
  AOM_T_NORM_RES_STD,
  AOM_T_AGENT_IDX,     /* int32 [n_agents][actor_in]  state index per actor input, -1 = pad (helper_states.py:286-317) */
  AOM_T_AGENT_ACT,     /* int32 [n_agents][actor_out] global action slot per actor output, -1 = pad (train_rpc.py:667-675) */
  AOM_T_AGENT_REWARD,  /* int32 [n_agents][2]  mode range [a0, a1) of the reward     (train_rpc.py:402-416)  */
  AOM_T_ACTOR_W1,      /* float [n_agents][hidden][ld(actor_in)]                      (model_rpc.py:78-84)   */
  AOM_T_ACTOR_B1,      /* float [n_agents][hidden] */
  AOM_T_ACTOR_W2,      /* float [n_agents][hidden][ld(hidden)] */
  AOM_T_ACTOR_B2,
  AOM_T_ACTOR_WH,      /* float [n_agents][2*actor_out][ld(hidden)]  mean rows then log-std rows */
  AOM_T_ACTOR_BH,      /* float [n_agents][2*actor_out] */
  AOM_T_GEO_PROJ,      /* float [nactu][ld(nactu)]    -(IF IF^T)^+ of the geometric controller (rtc_init.py:418-448) */
  AOM_T_GEO_SIFN,      /* float [nactu]        pupil sum of each influence row / number of pupil points           */
  AOM_T_DENOISER,      /* float [64452]        parameters of the per-subaperture denoiser, packed per layer as
                                               [input channel][tap][output channel] + bias (autoencoder_models.py:130-197) */
  AOM_T_DENOISER_TC,   /* [452 float][256000 B] the same denoiser for the tensor-core kernel: float parameters of the two
                                               CUDA-core layers and the scaled biases, then the fp16 hi / lo weight tiles of
                                               the four tcgen05 layers in streaming order (denoiser.py::pack_weights_tc) */
  AOM_T_COUNT
} aom_table;

/* Device buffers owned by the context (aom_get_buffer returns the device pointer and its element count). */
typedef enum aom_buffer {
  AOM_B_SCREEN = 0,    /* float [E][N][N] ring-buffered screen, index = layer           */
  AOM_B_RING_OX,       /* int32 [E]  physical column of logical column 0, index = layer */
  AOM_B_RING_OY,       /* int32 [E]                                                      */
  AOM_B_SLOPES,        /* float [E][ld(nslopes)]   rtc.get_slopes  (rtcCompass.py:104-114) */
  AOM_B_ERR,           /* float [E][ld(nactu)]     rtc.get_err                            */
  AOM_B_COM,           /* float [E][ld(nactu)]     rtc.get_command                        */
  AOM_B_VOLTS,         /* float [E][ld(nactu)]     rtc.get_voltages                       */
  AOM_B_BINCUBE,       /* float [E][nvalid][npix*npix]  (allocated on first use)          */
  AOM_B_PHASE,         /* float [E][n][n]               (allocated on first use)          */
  AOM_B_MODES,         /* float [E][ld(nmodes)]    scratch: last volts->modes product     */
  AOM_B_RES_MODES,     /* float [E][ld(nmodes)]    v2m . err of the last frame            */
  AOM_B_STATE,         /* float [E][ld(state_dim)]                                        */
  AOM_B_REWARD,        /* float [E][n_agents]                                             */
  AOM_B_ACTION,        /* float [E][ld(action_dim)]                                       */
  AOM_B_ACTION_MEAN,   /* float [E][ld(action_dim)]                                       */
  AOM_B_STREHL,        /* float [E][4]  SE, LE, phase variance, running mean variance     */
  AOM_B_GEO_COM,       /* float [E][ld(nactu)]     command of the geometric controller    */
  AOM_B_GEO_VOLTS,     /* float [E][ld(nactu)]     voltages on the mirrors it drives      */
  AOM_B_STREHL_GEO,    /* float [E][4]  as AOM_B_STREHL, for the target behind those mirrors */
  AOM_B_GEO_PROJ,      /* float [E][ld(nactu)]     IF (phi - <phi>): the phase projected on the influence functions */
  AOM_B_EXT_COUNT,     /* uint32 [E] extrusions since the environment's reset (its screen RNG counter), index = layer */
  AOM_B_COUNT
} aom_buffer;

/* Run-time switches (aom_set_option). */
typedef enum aom_option {
  AOM_OPT_WFS_PATH = 0, /* which Shack-Hartmann frame kernel serves the Nfft = 64 geometry */
  AOM_OPT_GEMM_PATH,    /* which GEMM kernel serves the env-batched contractions */
  AOM_OPT_TIME_WFS,     /* != 0: bracket every sensor-kernel launch with CUDA events (read with aom_wfs_time_ms) */
  AOM_OPT_GEO,          /* != 0: aom_step also runs the geometric controller every frame, as next_part_one does when
                           the parameter file lists one (rlSupervisor.py:1036-1046); needs the AOM_T_GEO_* tables */
  AOM_OPT_DENOISE,      /* != 0: aom_step keeps the detector cube and runs aom_denoise between the sensor frame and the
                           centroider, as next_part_one_integrator does when an autoencoder is configured
                           (rlSupervisor.py:968-979); needs AOM_T_DENOISER */
  AOM_OPT_PUPIL_PATH,   /* which kernels sweep the pupil-plane phase for aom_comp_strehl / aom_do_control_geo */
  AOM_OPT_KEEP_IMAGE,   /* != 0: aom_step keeps the detector cube of every frame in AOM_B_BINCUBE (d_bincube readers:
                           rlSupervisor.py:884-885, obtain_dataset_autoencoder.py:85-88) */
  AOM_OPT_STREHL,       /* != 0: aom_step evaluates the target Strehl every frame at AOM_OPT_STREHL_LAMBDA_NM, as
                           next_part_two does with compute_tar_psf=True (rlSupervisor.py:944-947).  1: the phase as traced
                           in the previous next_part_one, i.e. before this step's apply_control (the reference's default);
                           2: re-traced after apply_control (modification_online / "pure delay 0", rlSupervisor.py:936-940) */
  AOM_OPT_STREHL_LAMBDA_NM, /* target wavelength in nanometres for AOM_OPT_STREHL (default 1650) */
  AOM_OPT_EXTRUDE_PATH, /* which contraction serves the screen extrusion (aom_move_atmos / aom_reset) */
  AOM_OPT_STREHL_PEAK,  /* != 0: every aom_comp_strehl (and AOM_OPT_STREHL inside aom_step) behaves as with AOM_TAR_PEAK */
  AOM_OPT_PSF_NFFT,     /* size of the target's zero-padded focal grid (p_geom._ipupil: 2^ceil(log2(pupdiam) + 1)) */
  AOM_OPT_DENOISE_PATH, /* AOM_DENOISE_TCGEN05 (default when AOM_T_DENOISER_TC is uploaded) or AOM_DENOISE_SIMT */
  AOM_OPT_COUNT
} aom_option;
enum {
  AOM_EXTRUDE_I8 = 0,      /* exact integer contraction on tcgen05 (int8 digit planes, int32 accumulators, one rounding to
                              float32 per new pixel; default; extrude_i8.cuh) */
  AOM_EXTRUDE_FFMA = 1     /* float32 FFMA accumulation with round-to-nearest (round-1 kernel, cross-check path) */
};
enum {
  AOM_DENOISE_TCGEN05 = 0, /* e2, e3, d1, d2 as implicit GEMMs on tcgen05 (fp16 hi / lo operands, three products each), e1 and
                              d3 fused on the CUDA cores (denoise_tc.cuh); needs AOM_T_DENOISER_TC, else the next one runs */
  AOM_DENOISE_SIMT = 1     /* float32 FFMA kernel (denoise_kernels.cuh; cross-check path) */
};
enum {
  AOM_PUPIL_SWEEP = 0,     /* staged screen rows, one warp per strip of pupil rows (pitch-16 lattices; default; other
                              geometries fall back to AOM_PUPIL_PIXEL) */
  AOM_PUPIL_PIXEL = 1      /* one thread per pixel / one warp per row with plain global loads (cross-check path) */
};
enum {
  AOM_WFS_UMMA = 0,        /* both stages of the pruned DFT on tcgen05 / TMEM, eight subapertures per tensor-core tile, TMA-staged
                              screen tiles, three fp16 products per stage (fp32-grade; wfs_umma.cuh; serves the frames with noise or
                              a kept image under AOM_WFS_UMMA_WS too).  Geometries it does not cover fall back to
                              AOM_WFS_MMA_STAGED, then AOM_WFS_MMA_REG (aom_last_error says why) */
  AOM_WFS_UMMA_FAST = 1,   /* same, the stage-1 result handed to stage 2 as one rounded fp16 (slopes ~3e-5 relative) */
  AOM_WFS_SIMT = 2,        /* float32 shared-memory FFT on the FP32 pipe (cross-check path) */
  AOM_WFS_MMA_REG = 3,     /* round-1 generation 2: warp-level mma.sync DFT fed by plain global loads (any Nfft = 64 geometry) */
  AOM_WFS_MMA_STAGED = 4,  /* round-1 default: TMA-staged tiles + warp-level mma.sync DFT (cross-check / comparison path) */
  AOM_WFS_MMA_STAGED_FAST = 5, /* same, twiddle low parts dropped in stage 2 */
  AOM_WFS_UMMA_WS = 6      /* DEFAULT: the AOM_WFS_UMMA pipeline on specialised warps -- 8 field warps + 4 transform warps per
                              CTA, two stage-1 accumulators in TMEM (wfs_umma_ws.cuh); bit-identical results */
};

enum {
  AOM_GEMM_TCGEN05 = 0,    /* tensor cores (default): the controller's operator products (cmat, v2m, m2v) as exact integer
                              contractions (int8 digit planes on tcgen05 kind::i8, int32 accumulators, one rounding:
                              extrude_i8.cuh); the actors and everything else as three TF32 MMAs per product */
  AOM_GEMM_SIMT = 1,       /* float32 FFMA tiles (cross-check path) */
  AOM_GEMM_TF32 = 2        /* three TF32 MMAs per product everywhere (round-1 path: the tensor core truncates its float32
                              accumulator, ~3e-5 on K = 2400; comparison path) */
};

/* lifetime */
size_t aom_config_size(void);                       /* sizeof(aom_config) the library was built with (binding check) */
int aom_create(const aom_config* cfg, aom_ctx** out);
void aom_destroy(aom_ctx* ctx);
const char* aom_last_error(const aom_ctx* ctx);     /* ctx may be NULL for create-time errors */
/* Upload a table (host copy of nbytes).  The operators of the integer contractions (AOM_T_CMAT, AOM_T_V2M, AOM_T_M2V,
 * AOM_T_AB) must be finite: a NaN or an infinity in one of their valid columns returns AOM_ERR_INVALID and leaves the
 * table in force unchanged. */
int aom_set_table(aom_ctx* ctx, int table, int index, const void* host, size_t nbytes);
int aom_get_buffer(aom_ctx* ctx, int buffer, int index, void** dptr, size_t* count);
int aom_device_count_launches(const aom_ctx* ctx, uint64_t* n_launches);  /* kernels launched so far */
int aom_set_option(aom_ctx* ctx, int option, int value);
/* Synchronise the device and report asynchronous kernel-side errors (bounded waits that expired). */
int aom_check_device(aom_ctx* ctx);

/* RlSupervisor.reset (rlSupervisor.py:236-246): reseed + regenerate turbulence (2N extrusions per layer),
 * clear mirrors / integrator / delay line / histories.  seeds: host int64 [E]. */
int aom_reset(aom_ctx* ctx, const int64_t* seeds, void* stream);

/* Per-environment reset (the "autoreset" of vectorised environments): restart environments envs[0..n) (host int32,
 * distinct, 0 <= e < E) with seeds[0..n) (host int64) while the others run on.
 * - Each listed environment gets at once what aom_reset gives it: screens regenerated from its new seed (2N start-up
 *   extrusions per layer with its current amplitude and the sign of its current x wind, common or per-environment), ring
 *   origins, extrusion counters and wind accumulators at 0, and its rows of slopes, err, com, com1, volts, com_before,
 *   residual modes, every history slot, state, Strehl accumulators / figures and geometric controller buffers cleared.
 *   Set the new episode's conditions (aom_set_layer_amp / aom_set_layer_wind) before the call.
 * - Its next aom_step acts as the linear step that follows an aom_reset: its rl half-step is ignored (no action is
 *   injected, com stays 0, no Strehl is accumulated, reward 0) and the state it leaves is the s0 of a fresh episode
 *   (Gymnasium's next-step autoreset).  Called half-step by half-step: aom_rl_control skips the injection,
 *   aom_comp_strehl skips the environment and aom_state_end ends the status.
 * - Noise frames, actor decisions (exploration noise) and long-exposure counts of each environment count from its own
 *   reset.  From the call on, a listed environment computes bit for bit what it computes in a batch that was aom_reset
 *   with its new seed and given one linear step; every other environment computes what it would have without the call.
 * - AOM_ERR_INVALID: n < 0, an index out of range or listed twice.  AOM_ERR_STATE: no aom_reset yet.  n = 0: nothing.
 *   The round-1 sensor kernels (tensor_reg / tensor / tensor_fast) return AOM_ERR_UNSUPPORTED while environments are
 *   staggered, until the next aom_reset.  Waits for `stream`; cost about that of aom_reset for n = E, less for fewer. */
int aom_reset_envs(aom_ctx* ctx, int n, const int32_t* envs, const int64_t* seeds, void* stream);

/* AtmosCompass.move_atmos (atmosCompass.py:158-161) */
int aom_move_atmos(aom_ctx* ctx, void* stream);

/* AtmosCompass.set_wind / set_r0 (atmosCompass.py:79-135): new wind step (pixels / frame) and innovation
 * amplitude of one layer; a sign change of the wind needs no stencil upload (mirroring is index arithmetic). */
int aom_set_layer(aom_ctx* ctx, int layer, float deltax, float deltay, float amp);

/* AtmosCompass.set_r0 per environment (the reference changes r0 of its single simulator at run time,
 * train_rpc.py:429-449; a batch can hold one condition per environment): innovation amplitude of `layer` for every
 * environment, host float [E] (NULL: back to the layer's common amplitude).  The wind is set per environment by
 * aom_set_layer_wind. */
int aom_set_layer_amp(aom_ctx* ctx, int layer, const float* amp_host);

/* AtmosCompass.set_wind per environment (atmosCompass.py:79-135; the reference changes the wind of its single simulator
 * at run time, train_rpc.py:429-449): wind step (pixels / frame) of `layer` for every environment, host float [E] each
 * (NULL, NULL: back to the layer's common wind of aom_config.deltax / deltay and aom_set_layer).
 * - Setting per-environment winds starts every environment's accumulator from the layer's current common one: the
 *   screens do not jump mid-episode.  Every environment then sees exactly the extrusions, innovations and raytrace
 *   offsets it would see in a batch where every environment had its wind.
 * - aom_set_layer changes the common wind (and the amplitude) and leaves per-environment winds in force.
 * - Back on the common wind, the library returns to its uniform kernels as soon as every layer's accumulators agree
 *   over the batch, at the latest after the next aom_reset (whose start-up extrudes each environment in the direction
 *   of its own x wind).
 * - AOM_ERR_UNSUPPORTED when the pupil footprint of an environment leaves the screen.  The round-1 sensor kernels (wfs
 *   paths tensor_reg / tensor / tensor_fast) have no per-environment form: their frames return AOM_ERR_UNSUPPORTED
 *   ("per-environment wind is not implemented in the round-1 sensor kernels ...") while such winds are in force.
 * Waits for the device; not for the step path. */
int aom_set_layer_wind(aom_ctx* ctx, int layer, const float* deltax_host, const float* deltay_host);

/* WfsCompass.raytrace + compute_wfs_image fused (wfsCompass.py:334-343, sourceCompass.py:54-85).
 * flags: bit0 atmosphere, bit1 mirrors, bit2 keep image (writes AOM_B_BINCUBE), bit3 do not advance the frame counter
 * of the noise streams (a second look at the same frame, e.g. d_binimg_notnoisy of roket_generalized_rl.py:197). noise: sensor noise for
 * this frame (pass the common value of aom_set_wfs_noise, initially cfg.noise, for the configured one; with per-environment
 * noise in force any value >= 0 selects each environment's own).  Also leaves the centre-of-gravity slopes of the
 * frame for aom_do_centroids. */
int aom_comp_wfs_image(aom_ctx* ctx, int flags, float noise, void* stream);

/* WfsCompass.set_noise + the guide-star flux (geom_init.py:343-407): common sensor noise (<0 none, 0 photon, >0 photon
 * + read noise in e-) and photons per full subaperture and frame.  They start as aom_config.noise / nphotons; aom_step
 * draws its frames with them, and aom_comp_wfs_image scales its frames with this photon count.  AOM_ERR_INVALID for a
 * non-finite value or a photon count <= 0. */
int aom_set_wfs_noise(aom_ctx* ctx, float noise, float nphotons);

/* The same per environment (one guide-star magnitude and detector per environment of the batch): host float [E] each.
 * NULL returns that quantity to the common value; both NULL return to the uniform state.
 * - While per-environment noise is in force, aom_step and aom_comp_wfs_image with noise >= 0 draw each environment's
 *   frame with its own noise (the value passed then only means "noisy frame"); aom_comp_wfs_image with noise < 0 stays
 *   noise-free for every environment.  Every frame, and a kept image, is scaled by each environment's photon count.
 * - Every environment computes bit for bit what it computes in a batch configured with its values through aom_config.
 * - A frame in which no environment draws noise and no image is kept still runs the specialised-warp kernel
 *   (AOM_WFS_UMMA_WS); otherwise the per-environment form of the fused kernel (AOM_WFS_UMMA) serves it.
 * - Persists through aom_reset / aom_reset_envs: set the new episode's values before the reset call.
 * - AOM_ERR_INVALID for a non-finite entry or a photon count <= 0.  The round-1 sensor kernels (tensor_reg / tensor /
 *   tensor_fast) return AOM_ERR_UNSUPPORTED for a frame that would read per-environment sensor values.
 * Waits for the device; not for the step path. */
int aom_set_wfs_noise_env(aom_ctx* ctx, const float* noise_host, const float* nphotons_host);

/* Name of the kernel a noise-free aom_comp_wfs_image without kept image launches under the current AOM_OPT_WFS_PATH
 * ("wfs_frame_ws_kernel", "wfs_frame_umma_kernel", "wfs_frame_tma_kernel", "wfs_frame_mma_kernel" or "wfs_frame_kernel"), the
 * path's kernel also where the per-environment state makes that frame refused; when the staged kernel is not eligible for the
 * geometry, aom_last_error() says why. */
const char* aom_wfs_kernel(aom_ctx* ctx);

/* Mean device time (ms) of the sensor-kernel launches recorded since the last call (AOM_OPT_TIME_WFS; at most
 * AOM_WFS_TIMERS launches are kept); synchronises on the recorded events. */
int aom_wfs_time_ms(aom_ctx* ctx, float* mean_ms, int* count);

/* Materialise the pupil-plane phase seen by the sensor (wfs.get_wfs_phase) into AOM_B_PHASE. */
int aom_raytrace_wfs(aom_ctx* ctx, int flags, void* stream);

/* TargetCompass.comp_tar_image / comp_strehl / get_strehl (targetCompass.py:139-196) without the focal-plane image: the
 * phase of aom_raytrace_wfs is reduced over the pupil on the fly and AOM_B_STREHL = {SE, LE, variance, mean variance},
 * SE = |<exp(2 pi i phi / lambda)>|^2, the on-axis intensity ratio (the PSF peak of a tilt-free residual; equals the
 * Marechal value exp(-var (2 pi / lambda)^2) for small residuals), LE its mean over the accumulated frames.  flags as
 * aom_comp_wfs_image (bit0 atmosphere, bit1 mirrors); accumulate != 0 adds the frame to the long-exposure means.
 * The 2048^2 focal-plane PSF is not computed. */
#define AOM_TAR_GEO 0x100   /* flags bit: the target behind the geometric controller's mirrors (reads AOM_B_GEO_VOLTS,
                               writes AOM_B_STREHL_GEO) instead of the main ones */
#define AOM_TAR_PEAK 0x800  /* flags bit: Strehl from the brightest pixel of the PSF core (3 x 3 pixels of the reference's
                               Nfft focal grid, AOM_OPT_PSF_NFFT) with a three-point fit per axis, as comp_strehl(do_fit=True)
                               (targetCompass.py:139-196), instead of the on-axis pixel; the long exposure is the fit of
                               the accumulated core */
#define AOM_TAR_TRACE 0x200 /* flags bit: TargetCompass.raytrace only -- sweep the pupil now (current screens and voltages) and
                               keep the sums pending; nothing is published */
#define AOM_TAR_PUBLISH 0x400 /* flags bit: comp_tar_image / comp_strehl only -- publish (and accumulate) the pending sums of
                               the last AOM_TAR_TRACE.  Together they reproduce the reference's ordering when the mirrors
                               move between the target trace of next_part_one and the Strehl of next_part_two
                               (rlSupervisor.py:964-965, 944-947; "modification_online" re-traces after apply_control) */
int aom_comp_strehl(aom_ctx* ctx, int flags, float lambda_um, int accumulate, void* stream);
int aom_reset_strehl(aom_ctx* ctx, void* stream);     /* TargetCompass.reset_strehl */

/* Geometric controller (RlSupervisor.next_part_one_geo, rlSupervisor.py:989-1013; init_controller_geo,
 * rtc_init.py:418-448): aom_do_control_geo traces the target through the atmosphere and leaves
 * AOM_B_GEO_COM = -(IF IF^T)^+ IF (phi - <phi>), the least-squares mirror fit of the turbulent phase;
 * aom_apply_control_geo copies it to AOM_B_GEO_VOLTS (no latency: "geo pure delay 0").  The Strehl behind those
 * mirrors is aom_comp_strehl(flags | AOM_TAR_GEO). */
int aom_do_control_geo(aom_ctx* ctx, void* stream);
int aom_apply_control_geo(aom_ctx* ctx, void* stream);

/* Replace the detector image (RlSupervisor.autoencoder_denoising -> set_binimg, rlSupervisor.py:876-891):
 * device pointer to float [E][nvalid][npix*npix]; the next aom_do_centroids reads it. */
int aom_set_bincube(aom_ctx* ctx, const float* dcube, void* stream);

/* RlSupervisor.autoencoder_denoising (rlSupervisor.py:876-891) -> Autoencoder.predict (src/autoencoder/
 * autoencoder_models.py:199-240) for the per-subaperture CNN: every 16x16 spot of din [n_spots][256] through the six
 * layers in one fused kernel, result to dout.  din == NULL: the detector cube of the last frame (AOM_B_BINCUBE, needs
 * flag bit2 of aom_comp_wfs_image); dout == NULL: in place, and the next aom_do_centroids reads the denoised cube
 * (what set_binimg does in the reference).  n_spots is ignored when din == NULL. */
int aom_denoise(aom_ctx* ctx, const float* din, float* dout, long long n_spots, void* stream);

/* RtcCompass.do_centroids / do_control / set_command / apply_control (rtcCompass.py:557-563, 527-547, 463-473, 573-582) */
int aom_do_centroids(aom_ctx* ctx, void* stream);
/* RtcCompass.do_centroids_geom (rtcCompass.py; used by guardians/roket_generalized_rl.py:228, 246): AOM_B_SLOPES <- the mean
 * phase gradient per subaperture of the sensor-direction phase selected by flags (bit0 atmosphere, bit1 mirrors,
 * AOM_TAR_GEO: the geometric controller's mirrors), alpha = 0.206265 / subaperture size [m]. */
int aom_do_centroids_geom(aom_ctx* ctx, int flags, float alpha, void* stream);
/* err = -cmat.s and, loop closed, com += g err.  Non-finite inputs stay visible: an environment whose slopes (or, through
 * aom_rl_control, whose commands) hold a NaN or an infinity gets non-finite outputs in its own row and no other.  The
 * default tcgen05 path writes NaN to every output of that row; the SIMT path may give +-Inf instead. */
int aom_do_control(aom_ctx* ctx, void* stream);
int aom_set_command(aom_ctx* ctx, const float* dcom, int ld, void* stream);
int aom_apply_control(aom_ctx* ctx, int comp_voltage, void* stream);
int aom_set_gain(aom_ctx* ctx, float gain);     /* common gain; per-environment gains (aom_set_gain_env) stay in force */
/* RtcCompass.set_gain per environment (the reference tunes the integrator gain per parameter file, params.py): gain of
 * every environment's integrator, host float [E] (NULL: back to the common gain of aom_config.gain / aom_set_gain).
 * com += g[e] err in all three controller paths.  Persists through aom_reset / aom_reset_envs.  AOM_ERR_INVALID for a
 * non-finite entry.  Waits for the device; not for the step path. */
int aom_set_gain_env(aom_ctx* ctx, const float* gain_host);
int aom_set_loop(aom_ctx* ctx, int closed);       /* rtc.open_loop / close_loop (rtcCompass.py:116-142) */
int aom_reset_dm(aom_ctx* ctx, void* stream);     /* DmCompass.reset_dm */
int aom_set_dm_volts(aom_ctx* ctx, const float* dvolts, int ld, void* stream); /* DmCompass.set_command */

/* RlSupervisor.rl_control (rlSupervisor.py:713-733, 784-818): com <- m2v.(v2m.com + scatter(a * f)).
 * daction: device float [E][ld(action_dim)] (NULL: use AOM_B_ACTION). */
int aom_rl_control(aom_ctx* ctx, const float* daction, void* stream);

/* AoEnv.linear_step state assembly (ao_env.py:871-909): call aom_state_begin BEFORE the frame (captures the
 * command "before linear"), aom_state_end after do_control (projects, standardises, pushes history). */
int aom_state_begin(aom_ctx* ctx, void* stream);
int aom_state_end(aom_ctx* ctx, void* stream);

/* TrainerRPC.divide_rewards_for_agents (train_rpc.py:402-416): r[e][w] = -factor * mean((v2m.err)[a0:a1]^2) */
int aom_reward(aom_ctx* ctx, float factor, void* stream);

/* TrainerRPC.choose_action -> GaussianPolicy.sample(only_choosing_action=True) for every agent
 * (train_rpc.py:706-732, model_rpc.py:121-158).  eval_mode != 0: action = tanh(mean). */
int aom_actor_forward(aom_ctx* ctx, int eval_mode, void* stream);

/* One whole env-step: rl half-step (rl_control + apply_control + reward) and linear half-step
 * (move_atmos + WFS frame + centroids + control + state) -- TrainerRPC.env_step (train_rpc.py:633-648).
 * mode 0: actions from aom_actor_forward on the current state; 1: actions from AOM_B_ACTION; 2: integrator only.
 * mode | AOM_STEP_ATMOS_DONE: the caller has already advanced the turbulence for this step with aom_move_atmos (it
 * does not depend on the actions, so a host-in-the-loop caller can run it while the actions travel over PCIe). */
#define AOM_STEP_ATMOS_DONE 8
int aom_step(aom_ctx* ctx, int mode, int eval_mode, void* stream);

/* Generic device GEMM used by the path, exposed for the parity tests:
 * C[M][ldc] = A[M][lda] . B[N][ldb]^T (+ bias[N]) ; relu optional. */
int aom_gemm_tn(aom_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                int M, int N, int K, const float* bias, int relu, void* stream);

/* Sensor-noise sampler exposed for the parity tests: out[i] = noise(lam[i]) with pixel index i. */
int aom_pixel_noise(aom_ctx* ctx, const float* dlam, float* dout, int64_t n, float noise, int64_t seed,
                    uint32_t frame, uint32_t wfs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AOMARL_H */
