/* aogym.h -- C-ABI of libaogym.so: the B200 (sm_100a) implementation of the `AO-v0`
 * environment step path of payamparvizi/adaptive_optics_gym.
 *
 * The reference has no FFI: its hot path is pure Python calling hcipy (NumPy).  The entry
 * points below are what a binding for that path replaces, one handle per device holding N
 * lock-stepped environments:
 *
 *   aog_create / aog_set_table      <- AOEnv.__init__ + parameters_init + pupil_simulation +
 *                                      incoming_wavefront + DM_function + atmospheric_turbulence
 *                                      + fiber_coupling        (gym_AO/envs/AO_env.py:17-71,197-251,293-393)
 *   aog_set_screens / aog_generate_screens
 *                                   <- InfiniteAtmosphericLayer initial screen / layer.reset()
 *                                                              (AO_env.py:77,370)
 *   aog_reset[_host]                <- AOEnv.reset             (AO_env.py:74-103)
 *   aog_step[_host]                 <- AOEnv.step + reward_function (AO_env.py:106-153,468-503)
 *   aog_sh_configure + SH tables / aog_sh_step[_host]
 *                                   <- shack_hartmann_init / SH_step (AO_env.py:396-465,254-290)
 *   aog_get_field                   <- the fields AOEnv.render reads (AO_env.py:156-194)
 *
 * Conventions: every function returns 0 on success or a negative aog_status; nothing throws
 * across the ABI; aog_last_error() gives the message of the last failure on that handle.
 * All arrays are dense, row-major, env-major ([num_envs][...]).  Complex tables are
 * interleaved (re, im) doubles.  `stream` is a cudaStream_t passed as void*
 * (NULL = the CUDA default stream); the `*_host`
 * variants take HOST pointers, do the host<->device copies themselves and synchronise.
 * A handle is not thread-safe.  There is no CPU fallback: every entry point needs the GPU.
 */
#ifndef AOGYM_H
#define AOGYM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AOG_ABI_VERSION 2

#if defined(__GNUC__)
#define AOG_API __attribute__((visibility("default")))
#else
#define AOG_API
#endif

typedef struct aog_env aog_env; /* opaque */

typedef enum aog_status {
  AOG_OK = 0,
  AOG_ERR_INVALID = -1,   /* bad argument / configuration */
  AOG_ERR_CUDA = -2,      /* CUDA runtime failure (message in aog_last_error) */
  AOG_ERR_STATE = -3,     /* call sequence error (e.g. step before tables are set) */
  AOG_ERR_UNSUPPORTED = -4
} aog_status;

enum { AOG_ATM_QUASI_STATIC = 0, AOG_ATM_SEMI_DYNAMIC = 1, AOG_ATM_DYNAMIC = 2 };
enum { AOG_REW_STREHL_RATIO = 0, AOG_REW_SMF_SSIM = 1 };
enum { AOG_DTYPE_F32 = 0, AOG_DTYPE_F64 = 1 };
/* arithmetic of the step path:
 *   F64    FP64 everywhere (guaranteed parity)
 *   TENSOR tcgen05 DM GEMM + FP32 phase math + the fibre-arm matrix Fourier transform as split-fp16 tcgen05 GEMMs
 *   FUSED  tcgen05 DM GEMM + ONE fused kernel: the fibre coupling coefficients are inner products of the pupil
 *          field with the fibre modes propagated back to the pupil (G_j = M1^T (mode_j w) M2^T, FP64 on the host),
 *          so the screen is read once per step and neither the field nor the focal plane exists in HBM */
enum { AOG_PRECISION_F64 = 0, AOG_PRECISION_TENSOR = 1, AOG_PRECISION_FUSED = 2 };

/* Tables (host FP64 unless noted), sizes with Np pupil px/side, P = Np*Np, K modes, Nf focal
 * px/side, n obs px/side, J fibre modes, Ns stencil points. */
typedef enum aog_table {
  AOG_TABLE_APERTURE = 0,   /* [P]       0/1 aperture                       (AO_env.py:301) */
  AOG_TABLE_DM_MODES = 1,   /* [K][P]    influence functions / ptp          (AO_env.py:346-354) */
  AOG_TABLE_DM_GRAM = 2,    /* [K][K]    var(M a) = a^T G a                 (AO_env.py:120) */
  AOG_TABLE_MFT_FIB_1 = 3,  /* [Nf][Np]  complex, weights folded in         (AO_env.py:390) */
  AOG_TABLE_MFT_FIB_2 = 4,  /* [Np][Nf]  complex */
  AOG_TABLE_MFT_OBS_1 = 5,  /* [n][Np]   complex                            (AO_env.py:391) */
  AOG_TABLE_MFT_OBS_2 = 6,  /* [Np][n]   complex */
  AOG_TABLE_LP_MODES_W = 7, /* [J][Nf*Nf] fibre mode * focal weight          (AO_env.py:393,471) */
  AOG_TABLE_LP_PHASE = 8,   /* [J]       complex exp(i beta L) */
  AOG_TABLE_LP_GRAM = 9,    /* [J][J]    sum mode_j mode_k w */
  AOG_TABLE_AR_STENCIL = 10,/* [Ns]      int32 flat pixel indices           (AO_env.py:370) */
  AOG_TABLE_AR_A = 11,      /* [Np][Ns] */
  AOG_TABLE_AR_B = 12,      /* [Np][Np] */
  AOG_TABLE_SCR_C1 = 13,    /* [Np][Np]  spectral amplitudes, DFT scale     (AO_env.py:77) */
  AOG_TABLE_SCR_W1 = 14,    /* [Np][Np]  complex */
  AOG_TABLE_SCR_C2 = 15,    /* [N2][N2]  spectral amplitudes, fine scale */
  AOG_TABLE_SCR_W2 = 16,    /* [Np][N2]  complex */
  /* Shack-Hartmann integrator (SH_operation; AO_env.py:396-465), sizes from aog_sh_configure */
  AOG_TABLE_SH_MLA_PHASE = 17,   /* [P]        micro-lens array phase [rad] at lambda_wfs */
  AOG_TABLE_SH_FRESNEL = 18,     /* [Np][Np]   complex separable Fresnel operator C: E_out = C E C^T */
  AOG_TABLE_SH_PIX_OFFSETS = 19, /* [Nsub+1]   int32 CSR offsets of the pixels of each selected lenslet */
  AOG_TABLE_SH_PIX_INDEX = 20,   /* [npix]     int32 flat pixel index */
  AOG_TABLE_SH_PIX_X = 21,       /* [npix]     detector x coordinate of that pixel */
  AOG_TABLE_SH_PIX_Y = 22,       /* [npix] */
  AOG_TABLE_SH_OFFSET = 23,      /* [2][Nsub]  lenslet centre + reference slope (subtracted from the centroid) */
  AOG_TABLE_SH_RECON = 24,       /* [K][2 Nsub] reconstruction matrix */
  AOG_TABLE_SH_ACT0 = 25,        /* [K]        initial actuators of the SH mirror (broadcast to all envs) */
  AOG_TABLE_COUNT = 26
} aog_table;

enum { AOG_SH_NOISE_NONE = 0, AOG_SH_NOISE_POISSON = 1, AOG_SH_NOISE_INJECTED = 2 };

typedef enum aog_field {
  AOG_FIELD_SCREEN = 0,      /* [P]     achromatic screen S (phase = S / lambda), logical order */
  AOG_FIELD_PUPIL = 1,       /* [P]     complex pupil field after atmosphere + DM */
  AOG_FIELD_FOCAL = 2,       /* [Nf*Nf] complex focal field on the fibre plane */
  AOG_FIELD_FOCAL_POWER = 3, /* [Nf*Nf] |E|^2 w   (render panel 3)  */
  AOG_FIELD_OBS_POWER = 4,   /* [n*n]   photodetector power (render panel 4) */
  AOG_FIELD_ACTUATORS = 5,   /* [K]     DM actuators after normalisation */
  /* tensor-path intermediates of the last step (tests / debugging), hi + lo recombined: */
  AOG_FIELD_TC_PUPIL = 6,    /* [P]       complex, unit modulus x aperture */
  AOG_FIELD_TC_STAGE1 = 7,   /* [Nf*Np]   complex stage-1 product M1~ . E~ (unit-modulus twiddles) */
  AOG_FIELD_SH_IMAGE = 8,    /* [P]       noise-free Shack-Hartmann camera image for the current state */
  AOG_FIELD_SH_ACTUATORS = 9,/* [K]       actuators of the SH integrator's own mirror */
  AOG_FIELD_SH_IMAGE_TC = 10 /* [P]       the same camera image through the tensor-core kernels (tensor / fused handles) */
} aog_field;

typedef struct aog_config {
  int32_t abi_version;        /* AOG_ABI_VERSION */
  int32_t device;             /* CUDA ordinal */
  int32_t num_envs;           /* N lock-stepped environments on this device */
  int32_t num_pupil_pixels;   /* Np */
  int32_t num_focal_pixels;   /* Nf */
  int32_t obs_dim;            /* n  */
  int32_t num_modes;          /* K  */
  int32_t num_lp_modes;       /* J  */
  int32_t num_stencil;        /* Ns (0 unless dynamic) */
  int32_t num_screen_fine;    /* N2 (0 = no on-device screen synthesis) */
  int32_t atm_type;           /* AOG_ATM_* */
  int32_t rew_type;           /* AOG_REW_* */
  int32_t sh_operation;       /* step() applies the action unscaled (AO_env.py:115-116) */
  int32_t flat_mirror_start;  /* AO_env.py:79-80 */
  int32_t max_steps;          /* timesteps_per_episode */
  int32_t has_rew_threshold;
  int32_t precision;          /* AOG_PRECISION_* */
  int32_t env_id_base;        /* global id of env 0 (RNG stream = global env id) */
  double rew_threshold;
  double wavelength_wfs;
  double wavelength_sci;
  double delta_t;
  double velocity;            /* m/s along +x after the reference's coercion (AO_env.py:200-208) */
  double pupil_delta;         /* D / Np */
  double amp_fiber;           /* in-aperture amplitude of the unit-power wavefront */
  double sqrt_cn2;
  double strehl_scale;        /* strehl[%] = scale * |sum_ap exp(i phi_sci)|^2 */
  double obs_weight;          /* photodetector pixel area */
  double ssim_ref_peak;       /* 2.8 (AO_env.py:492) */
  double mft_norm_re;         /* 1 / (i lambda f) */
  double mft_norm_im;
  uint64_t seed;
} aog_config;

/* per-step outputs; any pointer may be NULL.  Device pointers for aog_step/aog_reset, host
 * pointers for the *_host variants. */
typedef struct aog_outputs {
  uint16_t* obs_f16;  /* [N][n*n]  IEEE half bits, RNE from FP64 (AO_env.py:103,153) */
  double* obs_f64;    /* [N][n*n]  before the float16 cast */
  double* reward;     /* [N] */
  double* power;      /* [N]      info["power"] = rew_fiber */
  double* strehl;     /* [N]      Strehl ratio in percent (strehl_ratio only) */
  double* ssim;       /* [N]      SSIM score (smf_ssim only) */
} aog_outputs;

typedef struct aog_counters {
  int64_t timestep;         /* global, never reset (AO_env.py:70,123) */
  int64_t timestep_render;  /* per episode (AO_env.py:83,124) */
  int64_t episode_no;       /* AO_env.py:149 */
  int64_t column_origin;    /* ring-buffer origin of the screens */
  int64_t extrusions;       /* extrusions done so far (Philox offset of the extrusion noise) */
  int64_t screen_draws;     /* von-Karman syntheses done so far (Philox offset of the screen generator) */
  int64_t sh_draws;         /* SH_step calls so far (Philox offset of the camera's photon noise) */
} aog_counters;

AOG_API const char* aog_version(void);
AOG_API int aog_create(const aog_config* cfg, aog_env** out);
AOG_API void aog_destroy(aog_env* env);
AOG_API const char* aog_last_error(const aog_env* env);

AOG_API int aog_set_table(aog_env* env, int which, const void* host, size_t count);

/* screens: [count][P] of `dtype`; src may be a host or a device pointer */
AOG_API int aog_set_screens(aog_env* env, const void* src, int dtype, int src_on_device, int first_env, int count);
AOG_API int aog_get_screens(aog_env* env, double* host_out, int first_env, int count);
/* new von-Karman screens for all envs from the on-device generator (semi_dynamic reset) */
AOG_API int aog_generate_screens(aog_env* env, void* stream);

/* per-env turbulence strength sqrt(Cn^2) [N] FP64 (host pointer), used by every later screen synthesis and
   extrusion; rescale != 0 also multiplies each env's current screen by new/old and refreshes its phase tiles.
   Values must be finite and > 0 (else AOG_ERR_INVALID, nothing changed).  aog_create starts every env at
   cfg.sqrt_cn2.  Stream-ordered on `stream`: no device synchronisation. */
AOG_API int aog_set_turbulence(aog_env* env, const double* sqrt_cn2_host, int rescale, void* stream);

/* number of column extrusions the next aog_step will perform (sizes `noise`) */
AOG_API int aog_next_extrusions(const aog_env* env);

AOG_API int aog_reset(aog_env* env, const aog_outputs* out_dev, void* stream);
AOG_API int aog_reset_host(aog_env* env, const aog_outputs* out_host);

/* actions: [N][K] of act_dtype.  noise: NULL (on-device Philox) or [N][n_ext][Np] FP64
 * standard normals consumed in order by this step's extrusions.  done_out: host int. */
AOG_API int aog_step(aog_env* env, const void* actions_dev, int act_dtype, const double* noise_dev,
             const aog_outputs* out_dev, int32_t* done_out, void* stream);
AOG_API int aog_step_host(aog_env* env, const void* actions_host, int act_dtype, const double* noise_host,
                  const aog_outputs* out_host, int32_t* done_out);

/* Shack-Hartmann integrator (AOEnv.SH_step, AO_env.py:254-290).  aog_sh_configure sizes the SH tables
 * (set them afterwards with aog_set_table).  noise_mode: AOG_SH_NOISE_*; `noisy_image` ([N][P] FP64, the
 * camera image AFTER photon noise) is read only in INJECTED mode.  action_out: [N][K] FP64. */
AOG_API int aog_sh_configure(aog_env* env, int num_sub, int num_pix, double amplitude, double weight_dt);
AOG_API int aog_sh_step(aog_env* env, int noise_mode, const double* noisy_image_dev, double* action_out_dev,
                        void* stream);
AOG_API int aog_sh_step_host(aog_env* env, int noise_mode, const double* noisy_image_host, double* action_out_host);

AOG_API int aog_get_counters(const aog_env* env, aog_counters* out);
AOG_API int aog_set_counters(aog_env* env, const aog_counters* in);
/* DM actuators [N][K] FP64 (state that survives reset when flat_mirror_start == 0) */
AOG_API int aog_get_actuators(aog_env* env, double* host_out);
AOG_API int aog_set_actuators(aog_env* env, const double* host_in);

/* actuators [N][K] FP64 of the Shack-Hartmann integrator's own mirror (AO_env.py:266,284-287,431); needs
 * aog_sh_configure */
AOG_API int aog_get_sh_actuators(aog_env* env, double* host_out);
AOG_API int aog_set_sh_actuators(aog_env* env, const double* host_in);

/* Re-key every random stream of the handle (extrusion noise, screen synthesis, photon noise) and restart their
 * draw counters: what AOEnv.reset(seed=s) does.  The reference ignores the seed (AO_env.py:74) and draws from
 * NumPy's global generator; here a seeded reset makes everything after it reproducible.  State (screens,
 * actuators, time) is untouched. */
AOG_API int aog_reseed(aog_env* env, uint64_t seed);

/* 0, or AOG_ERR_CUDA with aog_last_error naming the pipeline barrier that timed out (the tensor / fused kernels
 * trap instead of hanging; the flag lives in mapped host memory and stays readable after the trap) */
AOG_API int aog_health(aog_env* env);

AOG_API int aog_get_field(aog_env* env, int which, int env_index, double* host_out, size_t count);

/* test hook: n draws of the Shack-Hartmann camera's photon-noise sampler at rate lambda (Poisson below 1e6, rounded
 * normal above -- hcipy large_poisson, AO_env.py:274), Philox subsequence i for draw i; host_out [n] */
AOG_API int aog_debug_poisson(int device, double lambda, int n, uint64_t seed, double* host_out);

/* the FP32 photon-noise sampler of the tensor / fused handles' Shack-Hartmann camera (same test hook) */
AOG_API int aog_debug_poisson_f32(int device, double lambda, int n, uint64_t seed, double* host_out);

/* test hook: n Philox-4x32-10 blocks and the four standard normals the device makes of each.  philox != 0: words_in
 * holds n groups (counter[4], key[2]) and raw_out [n][4] receives the generator's words; philox == 0: words_in holds n
 * raw blocks [n][4] (raw_out unused).  generator 0: the extrusion noise and screen synthesis (aog_normals4), 1: the
 * Shack-Hartmann camera (normals4).  normals_out [n][4] */
AOG_API int aog_debug_normals(int device, int generator, int philox, int n, const uint32_t* words_in, uint32_t* raw_out,
                              float* normals_out);

/* kernels launched by this handle since creation (bench.py's gpu_launches) */
AOG_API int64_t aog_launch_count(const aog_env* env);
/* environments processed per kernel sequence (num_envs is walked in chunks of this size) */
AOG_API int aog_chunk_size(const aog_env* env);
/* device time [ms] of the dominant (MFT) kernel sequence of the LAST chunk of the last step,
 * CUDA events on the launch stream; negative if timing is disabled */
AOG_API int aog_set_timing(aog_env* env, int enabled);
AOG_API double aog_last_mft_ms(aog_env* env);
/* tensor / fused paths: the phase kernel (fused path: the whole optics kernel) and the two MFT stages (0 on the fused
 * path) of the last timed chunk, milliseconds */
AOG_API int aog_last_kernel_ms(aog_env* env, double* field_ms, double* stage1_ms, double* stage2_ms);

/* more device times [ms] of the last timed step (negative = not recorded), out_ms[n >= 7]:
 *   [0] all column extrusions of the last aog_step, [1] how many there were,
 *   [2..6] the tensor-core Shack-Hartmann step's kernels (last chunk): phase, fold, first product, second product, camera */
AOG_API int aog_last_timings(aog_env* env, double* out_ms, int n);

#ifdef __cplusplus
}
#endif
#endif /* AOGYM_H */
