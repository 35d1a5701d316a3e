// Shared declarations of libaogym (sm_100a).  See include/aogym.h for the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>
#include "aogym.h"

#define AOG_MAX_LP 8       // guided fibre modes kept in registers (reference config: 3)
#define AOG_MAX_OBS 16     // obs_dim upper bound (reference uses 2..5)

// ---- ownership of the handle's CUDA resources: each is released once, by its owner's destructor ----
// One cudaMalloc (device) or cudaHostAlloc (pinned host) allocation.  It converts to T* so that kernel arguments and
// pointer arithmetic take it as a plain pointer.
template <typename T, bool PINNED = false>
class CudaArray {
 public:
  CudaArray() = default;
  CudaArray(CudaArray&& o) noexcept : p_(std::exchange(o.p_, nullptr)) {}
  CudaArray& operator=(CudaArray&& o) noexcept { std::swap(p_, o.p_); return *this; }
  ~CudaArray() { reset(); }
  T* get() const { return p_; }
  operator T*() const { return p_; }
  void reset() {
    if (p_) PINNED ? cudaFreeHost(p_) : cudaFree(p_);
    p_ = nullptr;
  }
  // frees the old array first; a count of 0 leaves the array empty
  cudaError_t alloc(size_t count, unsigned host_flags = cudaHostAllocDefault) {
    reset();
    if (count == 0) return cudaSuccess;
    const cudaError_t e = PINNED ? cudaHostAlloc((void**)&p_, count * sizeof(T), host_flags)
                                 : cudaMalloc((void**)&p_, count * sizeof(T));
    if (e != cudaSuccess) p_ = nullptr;
    return e;
  }
  int alloc(aog_env* env, size_t count);   // the same, the error reported through env->err (defined below)
 private:
  T* p_ = nullptr;
};
template <typename T> using DevArray = CudaArray<T>;
template <typename T> using PinnedArray = CudaArray<T, true>;

template <typename H, cudaError_t (*DESTROY)(H)>
struct Destroy { void operator()(H h) const { DESTROY(h); } };
using StreamPtr = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, Destroy<cudaStream_t, cudaStreamDestroy>>;
using EventPtr = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, Destroy<cudaEvent_t, cudaEventDestroy>>;
using GraphExecPtr = std::unique_ptr<std::remove_pointer_t<cudaGraphExec_t>, Destroy<cudaGraphExec_t, cudaGraphExecDestroy>>;
// creates a stream / event / graph exec into its owner: cuda_create(env->ev0, cudaEventCreateWithFlags, cudaEventDefault)
template <typename Owner, typename Fn, typename... Args>
cudaError_t cuda_create(Owner& owner, Fn fn, Args... args) {
  typename Owner::pointer h = nullptr;
  const cudaError_t e = fn(&h, args...);
  owner.reset(e == cudaSuccess ? h : nullptr);
  return e;
}

// the state of the tensor / fused paths, defined (with its deleter) in tensor_path.cu
struct TensorState;
struct TensorStateDeleter { void operator()(TensorState* ts) const; };

struct aog_env {
  aog_config cfg{};
  int P = 0, NF2 = 0, n2 = 0;
  std::string err;
  bool have[AOG_TABLE_COUNT] = {};

  // ---- tables (device) ----
  DevArray<double> t_aperture;      // [P]
  DevArray<double> t_modes;         // [K][P]
  DevArray<double> t_gram;          // [K][K]
  DevArray<double2> t_m1f;          // [Nf][Np]
  DevArray<double2> t_m2f;          // [Np][Nf]
  DevArray<double2> t_m1o;          // [n][Np]
  DevArray<double2> t_m2o;          // [Np][n]
  DevArray<double> t_lpw;           // [J][Nf*Nf]
  DevArray<double2> t_lpphase;      // [J]
  DevArray<double> t_lpgram;        // [J][J]
  DevArray<int> t_stencil;          // [Ns] flat pixel indices in GATHER order (sorted by column, then row)
  DevArray<int> t_stencil_perm;     // [Ns] gather position -> index into the uploaded (row-major sorted) stencil
  DevArray<double> t_arA;           // [Np][Ns] as uploaded
  DevArray<double> t_arB;           // [Np][Np] as uploaded
  DevArray<double> t_arW;           // [(Ns+Np)][Np] = [A^T ; B^T]  (GEMM operand)
  DevArray<double> t_arW_rev;       // the same with the rows of the two full stencil columns reversed (k_ar_step<DIRECT>, +x)
  DevArray<int> t_ar_tail;          // [Ns - 2 Np] (x | y << 16) of the stencil's tail pixels, gather order
  bool ar_direct = false;          // the stencil is [column 0 | column 1 | tail]: k_ar_step reads the screens in place
  DevArray<double> t_scrC1;         // [Np][Np]
  DevArray<double2> t_scrW1;        // [Np][Np]
  DevArray<double2> t_scrW1T;       // transpose
  DevArray<double> t_scrC2;         // [N2][N2]
  DevArray<double2> t_scrW2;        // [Np][N2]
  DevArray<double2> t_scrW2T;       // [N2][Np]
  DevArray<double2> t_scr_sh;       // [Np] W1[0][k]: W1[x][k] = sh[k] w^(x k) (a shifted DFT matrix) -> FFT synthesis (fft240.cuh)
  DevArray<double2> t_scr_tw;       // [240] w^j = exp(2 pi i j / 240)
  bool scr_fft = false;

  // ---- Shack-Hartmann tables / state ----
  int sh_num_sub = 0, sh_num_pix = 0;
  double sh_amplitude = 0.0, sh_weight_dt = 0.0;
  DevArray<double> t_sh_mla;        // [P]
  DevArray<double2> t_sh_C;         // [Np][Np]
  DevArray<double2> t_sh_CT;        // transpose
  // Centrosymmetric Fresnel operator (C[N-1-i][N-1-j] = C[i][j], checked at upload): C acts separately on the even
  // and odd parts of a vector, so E_out = C E C^T splits into four (N/2)^3 products, half the work.
  // t_sh_Cf = {Ce, Co, Ce^T, Co^T}, each [N/2][N/2], Ce/o[i][j] = (C[i][j] +- C[i][N-1-j]) / 2
  // von-Karman synthesis S = Re(W X W^T) in real arithmetic when the rows of W come in conjugate pairs
  // (W[N-1-x][k] = conj(W[x][k]): symmetric pupil coordinates; checked at upload).  Per scale s (0: FFT grid, 1: the
  // oversampled low-frequency grid): t_scrWst[s] = [Re W_top ; Im W_top] (N x Nk), t_scrWrT / t_scrWiT = their
  // transposes (Nk x N/2).  2.7x fewer flops than the two complex GEMMs, and real GEMMs run on the FP64 tensor cores.
  bool scr_sym[2] = {false, false};
  DevArray<double> t_scrWst[2];
  DevArray<double> t_scrWrT[2];
  DevArray<double> t_scrWiT[2];
  bool sh_fold = false;
  DevArray<double2> t_sh_Cf[4];
  DevArray<int> t_sh_off;           // [Nsub+1]
  DevArray<int> t_sh_pix;           // [npix]
  DevArray<double> t_sh_px;         // [npix]
  DevArray<double> t_sh_py;         // [npix]
  DevArray<double> t_sh_offset;     // [2][Nsub]
  DevArray<double> t_sh_recon;      // [K][2 Nsub]
  DevArray<double> t_sh_act0;       // [K]
  DevArray<double> act_sh;          // [B][K] actuators of the SH integrator's mirror
  DevArray<double> o_action;        // [B][K] device staging for aog_sh_step_host
  DevArray<double> sh_noisy_in;     // [B][P] staging for an injected camera image
  int64_t sh_draws = 0;

  // ---- per-env state (device) ----
  DevArray<double> screens;         // [B][Np x][Np y] COLUMN-major (a pupil column is contiguous: the extrusion reads and
                                   // writes whole columns), ring-buffered along x (column_origin)
  DevArray<double> act;             // [B][K] DM actuators (after normalisation)
  DevArray<double> sqrt_cn2;        // [2 B] turbulence strength sqrt(Cn^2) of each env (read by the screen synthesis and
                                   // the extrusion noise), then the factors of the last aog_set_turbulence rescale
  std::vector<double> sqrt_cn2_host;   // [B] host copy of the first half (the old values of a rescale)

  // ---- scratch for one chunk of envs ----
  int chunk = 0;
  DevArray<double2> bufA;           // [chunk][P]              pupil field E
  DevArray<double2> bufB;           // [chunk][Np*max(Nf,Np)]  stage-1 product T
  DevArray<double2> bufC;           // [chunk][max(Nf*Nf,P)]   focal field F
  DevArray<double2> bufR;           // [chunk][Np*n]           obs-arm row products
  DevArray<double2> coef;           // [chunk][J]              fibre-mode coefficients
  DevArray<double2> strehl_part;    // [chunk][strehl_blocks]
  int strehl_blocks = 0;
  DevArray<double> arZ;             // [chunk][Ns+Np]
  DevArray<double> arNZ;            // [arNZ_cap extrusions][chunk][Np] scaled normals of one step (k_ar_noise)
  int arNZ_cap = 0;
  DevArray<double> act_in;          // [B][K] staging of raw actions (f64-sized)
  DevArray<double> noise_in;        // staging for injected noise
  size_t noise_in_cap = 0;
  // device-side outputs used by the *_host variants: not owned, slices of o_pack
  uint16_t* o_obs16 = nullptr; double* o_obs64 = nullptr; double* o_reward = nullptr;
  double* o_power = nullptr; double* o_strehl = nullptr; double* o_ssim = nullptr;
  DevArray<char> o_pack; size_t o_pack_bytes = 0;   // the six arrays above are slices of this one allocation (one D2H copy)
  // pinned host staging
  PinnedArray<char> h_pinned; size_t h_pinned_cap = 0;
  // small batches (<= 256 envs, static atmosphere): the host-buffer step (H2D actions, kernels, D2H outputs) is
  // captured once in a CUDA graph and relaunched -- one driver call instead of ~8 launches + copies
  PinnedArray<double> h_act;        // pinned staging of the actions (the graph's H2D source)
  GraphExecPtr step_graph;
  int graph_dtype = -1, graph_warm = 0, graph_launches = 0;
  bool graph_failed = false;

  // ---- counters (host; all envs run in lock-step) ----
  aog_counters cnt{};
  int64_t launches = 0;
  int64_t screen_draws = 0;        // von-Karman syntheses so far (Philox offset domain)
  std::unique_ptr<TensorState, TensorStateDeleter> tensor;   // tensor / fused precision only
  int32_t* phase_tiles = nullptr;   // not owned: TensorState::hwt (tiled fixed-point phase) for k_ar_step's epilogue, else null
  double phase_tiles_unit = 0.0;    // fixed-point units per half-turn (PHI_ONE)
  StreamPtr own_stream;
  // configs[3]: the column extrusions of step t only wait for the PHASE kernel of SH_step t (the last reader of the
  // screens / phase tiles), so they run on a side stream under SH_step's remaining, HBM-bound kernels
  StreamPtr side_stream;
  EventPtr ev_sh_phase, ev_ext_done;
  bool sh_phase_pending = false;
  cudaStream_t sh_phase_stream = nullptr;   // not owned: the caller's stream of that SH_step
  bool timing = false;
  EventPtr ev0, ev1, evf, evm;      // evf: before the field kernel, evm: between the MFT stages
  bool ev_valid = false;
  // aog_last_timings: [0,1] around the extrusions of the last step; [2..7] boundaries of the five kernels of the
  // tensor-core Shack-Hartmann step (last chunk)
  EventPtr tev[8];
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

template <typename T, bool PINNED>
int CudaArray<T, PINNED>::alloc(aog_env* env, size_t count) { AOG_CUDA(alloc(count)); return AOG_OK; }

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
