// Shared declarations of libaogym (sm_100a).  See include/aogym.h for the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "aogym.h"

#define AOG_MAX_LP 8       // guided fibre modes kept in registers (reference config: 3)
#define AOG_MAX_OBS 16     // obs_dim upper bound (reference uses 2..5)

struct aog_env {
  aog_config cfg{};
  int P = 0, NF2 = 0, n2 = 0;
  std::string err;
  bool have[AOG_TABLE_COUNT] = {};

  // ---- tables (device) ----
  double* t_aperture = nullptr;    // [P]
  double* t_modes = nullptr;       // [K][P]
  double* t_gram = nullptr;        // [K][K]
  double2* t_m1f = nullptr;        // [Nf][Np]
  double2* t_m2f = nullptr;        // [Np][Nf]
  double2* t_m1o = nullptr;        // [n][Np]
  double2* t_m2o = nullptr;        // [Np][n]
  double* t_lpw = nullptr;         // [J][Nf*Nf]
  double2* t_lpphase = nullptr;    // [J]
  double* t_lpgram = nullptr;      // [J][J]
  int* t_stencil = nullptr;        // [Ns] flat pixel indices in GATHER order (sorted by column, then row)
  int* t_stencil_perm = nullptr;   // [Ns] gather position -> index into the uploaded (row-major sorted) stencil
  double* t_arA = nullptr;         // [Np][Ns] as uploaded
  double* t_arB = nullptr;         // [Np][Np] as uploaded
  double* t_arW = nullptr;         // [(Ns+Np)][Np] = [A^T ; B^T]  (GEMM operand)
  double* t_arW_rev = nullptr;     // the same with the rows of the two full stencil columns reversed (k_ar_step<DIRECT>, +x)
  int* t_ar_tail = nullptr;        // [Ns - 2 Np] (x | y << 16) of the stencil's tail pixels, gather order
  bool ar_direct = false;          // the stencil is [column 0 | column 1 | tail]: k_ar_step reads the screens in place
  double* t_scrC1 = nullptr;       // [Np][Np]
  double2* t_scrW1 = nullptr;      // [Np][Np]
  double2* t_scrW1T = nullptr;     // transpose
  double* t_scrC2 = nullptr;       // [N2][N2]
  double2* t_scrW2 = nullptr;      // [Np][N2]
  double2* t_scrW2T = nullptr;     // [N2][Np]
  double2* t_scr_sh = nullptr;     // [Np] W1[0][k]: W1[x][k] = sh[k] w^(x k) (a shifted DFT matrix) -> FFT synthesis (fft240.cuh)
  double2* t_scr_tw = nullptr;     // [240] w^j = exp(2 pi i j / 240)
  bool scr_fft = false;

  // ---- Shack-Hartmann tables / state ----
  int sh_num_sub = 0, sh_num_pix = 0;
  double sh_amplitude = 0.0, sh_weight_dt = 0.0;
  double* t_sh_mla = nullptr;      // [P]
  double2* t_sh_C = nullptr;       // [Np][Np]
  double2* t_sh_CT = nullptr;      // transpose
  // Centrosymmetric Fresnel operator (C[N-1-i][N-1-j] = C[i][j], checked at upload): C acts separately on the even
  // and odd parts of a vector, so E_out = C E C^T splits into four (N/2)^3 products, half the work.
  // t_sh_Cf = {Ce, Co, Ce^T, Co^T}, each [N/2][N/2], Ce/o[i][j] = (C[i][j] +- C[i][N-1-j]) / 2
  // von-Karman synthesis S = Re(W X W^T) in real arithmetic when the rows of W come in conjugate pairs
  // (W[N-1-x][k] = conj(W[x][k]): symmetric pupil coordinates; checked at upload).  Per scale s (0: FFT grid, 1: the
  // oversampled low-frequency grid): t_scrWst[s] = [Re W_top ; Im W_top] (N x Nk), t_scrWrT / t_scrWiT = their
  // transposes (Nk x N/2).  2.7x fewer flops than the two complex GEMMs, and real GEMMs run on the FP64 tensor cores.
  bool scr_sym[2] = {false, false};
  double* t_scrWst[2] = {nullptr, nullptr};
  double* t_scrWrT[2] = {nullptr, nullptr};
  double* t_scrWiT[2] = {nullptr, nullptr};
  bool sh_fold = false;
  double2* t_sh_Cf[4] = {nullptr, nullptr, nullptr, nullptr};
  int* t_sh_off = nullptr;         // [Nsub+1]
  int* t_sh_pix = nullptr;         // [npix]
  double* t_sh_px = nullptr;       // [npix]
  double* t_sh_py = nullptr;       // [npix]
  double* t_sh_offset = nullptr;   // [2][Nsub]
  double* t_sh_recon = nullptr;    // [K][2 Nsub]
  double* t_sh_act0 = nullptr;     // [K]
  double* act_sh = nullptr;        // [B][K] actuators of the SH integrator's mirror
  double* o_action = nullptr;      // [B][K] device staging for aog_sh_step_host
  double* sh_noisy_in = nullptr;   // [B][P] staging for an injected camera image
  int64_t sh_draws = 0;

  // ---- per-env state (device) ----
  double* screens = nullptr;       // [B][Np x][Np y] COLUMN-major (a pupil column is contiguous: the extrusion reads and
                                   // writes whole columns), ring-buffered along x (column_origin)
  double* act = nullptr;           // [B][K] DM actuators (after normalisation)
  double* sqrt_cn2 = nullptr;      // [2 B] turbulence strength sqrt(Cn^2) of each env (read by the screen synthesis and
                                   // the extrusion noise), then the factors of the last aog_set_turbulence rescale
  std::vector<double> sqrt_cn2_host;   // [B] host copy of the first half (the old values of a rescale)

  // ---- scratch for one chunk of envs ----
  int chunk = 0;
  double2* bufA = nullptr;         // [chunk][P]              pupil field E
  double2* bufB = nullptr;         // [chunk][Np*max(Nf,Np)]  stage-1 product T
  double2* bufC = nullptr;         // [chunk][max(Nf*Nf,P)]   focal field F
  double2* bufR = nullptr;         // [chunk][Np*n]           obs-arm row products
  double2* coef = nullptr;         // [chunk][J]              fibre-mode coefficients
  double2* strehl_part = nullptr;  // [chunk][strehl_blocks]
  int strehl_blocks = 0;
  double* arZ = nullptr;           // [chunk][Ns+Np]
  double* arNZ = nullptr;          // [arNZ_cap extrusions][chunk][Np] scaled normals of one step (k_ar_noise)
  int arNZ_cap = 0;
  void* act_in = nullptr;          // [B][K] staging of raw actions (f64-sized)
  double* noise_in = nullptr;      // staging for injected noise
  size_t noise_in_cap = 0;
  // device-side outputs used by the *_host variants
  uint16_t* o_obs16 = nullptr; double* o_obs64 = nullptr; double* o_reward = nullptr;
  double* o_power = nullptr; double* o_strehl = nullptr; double* o_ssim = nullptr;
  char* o_pack = nullptr; size_t o_pack_bytes = 0;   // the six arrays above are slices of this one allocation (one D2H copy)
  // pinned host staging
  void* h_pinned = nullptr; size_t h_pinned_cap = 0;
  // small batches (<= 256 envs, static atmosphere): the host-buffer step (H2D actions, kernels, D2H outputs) is
  // captured once in a CUDA graph and relaunched -- one driver call instead of ~8 launches + copies
  void* h_act = nullptr;                // pinned staging of the actions (the graph's H2D source)
  cudaGraphExec_t step_graph = nullptr;
  int graph_dtype = -1, graph_warm = 0, graph_launches = 0;
  bool graph_failed = false;

  // ---- counters (host; all envs run in lock-step) ----
  aog_counters cnt{};
  int64_t launches = 0;
  int64_t screen_draws = 0;        // von-Karman syntheses so far (Philox offset domain)
  void* tensor_state = nullptr;     // TensorState (tensor_path.cu) when precision == TENSOR
  int32_t* phase_tiles = nullptr;   // TensorState::hwt (tiled fixed-point phase) for k_ar_step's epilogue, else null
  double phase_tiles_unit = 0.0;    // fixed-point units per half-turn (PHI_ONE)
  cudaStream_t own_stream = nullptr;
  // configs[3]: the column extrusions of step t only wait for the PHASE kernel of SH_step t (the last reader of the
  // screens / phase tiles), so they run on a side stream under SH_step's remaining, HBM-bound kernels
  cudaStream_t side_stream = nullptr;
  cudaEvent_t ev_sh_phase = nullptr, ev_ext_done = nullptr;
  bool sh_phase_pending = false;
  cudaStream_t sh_phase_stream = nullptr;
  bool timing = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evf = nullptr, evm = nullptr;   // evf: before the field kernel, evm: between the MFT stages
  bool ev_valid = false;
  // aog_last_timings: [0,1] around the extrusions of the last step; [2..7] boundaries of the five kernels of the
  // tensor-core Shack-Hartmann step (last chunk)
  cudaEvent_t tev[8] = {};
  bool tev_ext_valid = false, tev_sh_valid = false;
  int last_extrusions = 0;
};

// tensor_path.cu: appends the code of a timed-out pipeline barrier (if one fired) to env->err -- a trap surfaces as a
// generic sticky CUDA error on the next call, and this is what says which barrier it was
void aog_tensor_annotate_error(aog_env* env);

#define AOG_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      env->err = std::string(#call) + ": " + cudaGetErrorString(_e);                    \
      aog_tensor_annotate_error(env);                                                   \
      return AOG_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

// Every C-ABI entry point runs on the handle's device and restores the caller's current device on every return
// path (torch reads the current device through cudaGetDevice: a handle on device 1 must not move the caller there).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) {
      err = cudaSetDevice(dev);
      switched = err == cudaSuccess;
    }
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define AOG_DEVICE(dev)                                                                  \
  DeviceGuard _aog_guard(dev);                                                           \
  if (_aog_guard.err != cudaSuccess) {                                                   \
    env->err = std::string("cudaSetDevice: ") + cudaGetErrorString(_aog_guard.err);      \
    return AOG_ERR_CUDA;                                                                 \
  }

#define AOG_FAIL(code, msg) \
  do { env->err = (msg); return (code); } while (0)

#define AOG_LAUNCH_CHECK()                                   \
  do {                                                       \
    env->launches++;                                         \
    AOG_CUDA(cudaGetLastError());                            \
  } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
