// libaogym: C-ABI + host orchestration of the AO-v0 step path on B200 (sm_100a).
// See include/aogym.h for the contract and the reference lines each entry point replaces.
#include "common.cuh"
#include "kernels_f64.cuh"
#include "tensor_path.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

namespace {

template <typename T>
int dev_alloc(aog_env* env, T** p, size_t count) {
  if (*p) { cudaFree(*p); *p = nullptr; }
  if (count == 0) return AOG_OK;
  AOG_CUDA(cudaMalloc((void**)p, count * sizeof(T)));
  return AOG_OK;
}

int ensure_pinned(aog_env* env, size_t bytes) {
  if (bytes <= env->h_pinned_cap) return AOG_OK;
  if (env->h_pinned) cudaFreeHost(env->h_pinned);
  env->h_pinned = nullptr;
  env->h_pinned_cap = 0;
  AOG_CUDA(cudaMallocHost(&env->h_pinned, bytes));
  env->h_pinned_cap = bytes;
  return AOG_OK;
}

bool tables_ready(aog_env* env) {
  static const int need[] = {AOG_TABLE_APERTURE, AOG_TABLE_DM_MODES, AOG_TABLE_DM_GRAM, AOG_TABLE_MFT_FIB_1,
                             AOG_TABLE_MFT_FIB_2, AOG_TABLE_MFT_OBS_1, AOG_TABLE_MFT_OBS_2, AOG_TABLE_LP_MODES_W,
                             AOG_TABLE_LP_PHASE, AOG_TABLE_LP_GRAM};
  for (int t : need)
    if (!env->have[t]) { env->err = "table " + std::to_string(t) + " not set"; return false; }
  if (env->cfg.atm_type == AOG_ATM_DYNAMIC && env->cfg.velocity != 0.0)
    for (int t : {AOG_TABLE_AR_STENCIL, AOG_TABLE_AR_A, AOG_TABLE_AR_B})
      if (!env->have[t]) { env->err = "AR table " + std::to_string(t) + " not set"; return false; }
  return true;
}

int64_t center_px(const aog_env* env, int64_t timestep) {
  // hcipy evolve_until: round(velocity * t / delta), np.round = round-half-even
  const double t = (double)timestep * env->cfg.delta_t;
  const double c = env->cfg.velocity * t;
  return (int64_t)std::nearbyint(c / env->cfg.pupil_delta);
}

// the FP64 tensor-core GEMMs keep their cp.async ring in opt-in dynamic shared memory
int dmma_configure(aog_env* env) {
  static std::atomic<bool> done_on[64];    // function attributes are per device: one flag per device ordinal
  std::atomic<bool>& done = done_on[env->cfg.device & 63];
  if (done.load(std::memory_order_acquire)) return AOG_OK;
  AOG_CUDA(cudaFuncSetAttribute(k_ar_step<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AR_SMEM));
  AOG_CUDA(cudaFuncSetAttribute(k_ar_step<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, AR_SMEM + 4096 * 4));
  AOG_CUDA(cudaFuncSetAttribute(k_dgemm_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, DmmaCfg<1>::SMEM));
  AOG_CUDA(cudaFuncSetAttribute(k_scr_fft_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, FFT_SMEM));
  AOG_CUDA(cudaFuncSetAttribute(k_scr_fft_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, FFT_SMEM));
  done.store(true, std::memory_order_release);
  return AOG_OK;
}

// ---- one column extrusion for all envs -------------------------------------------------
int extrude_once(aog_env* env, bool positive, const double* noise_dev, long long noise_stride, cudaStream_t st) {
  const aog_config& c = env->cfg;
  const int Np = c.num_pupil_pixels, Ns = c.num_stencil, B = c.num_envs;
  const int flipped = positive ? 1 : 0;   // +x drift = hcipy 'right' = extrude on the rotated screen
  const int org = (int)env->cnt.column_origin;
  const int phys = positive ? org : (org - 1 + Np) % Np;
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    dim3 g1(cdiv(Ns + Np, 256), nB);
    k_ar_gather<<<g1, 256, 0, st>>>(env->screens, env->t_stencil, noise_dev, env->arZ, env->P, Np, Ns, e0, org,
                                    flipped, env->sqrt_cn2, noise_stride, c.seed, (unsigned long long)c.env_id_base,
                                    (unsigned long long)env->cnt.extrusions);
    AOG_LAUNCH_CHECK();
    // GEMM with the scatter into the ring slot (and the phase-tile refresh of the tensor / fused paths) in its epilogue
    dim3 g2(cdiv(Np, 64), cdiv(nB, AR_TM));
    { int rc = dmma_configure(env); if (rc) return rc; }
    k_ar_step<false><<<g2, AR_THREADS, AR_SMEM, st>>>(env->arZ, env->t_arW, env->screens, env->phase_tiles, nB, Np, Ns + Np, env->P, e0, phys,
                                  flipped, 1.0 / (c.wavelength_wfs * 3.14159265358979323846), env->phase_tiles_unit, ArDirect{});
    AOG_LAUNCH_CHECK();
  }
  env->cnt.column_origin = positive ? (org + 1) % Np : phys;
  env->cnt.extrusions++;
  return AOG_OK;
}

// ---- all the column extrusions of one step, the stencil read in place (k_ar_step<DIRECT>) --------------------
// Envs are independent, so the loop runs chunk by chunk: one k_ar_noise launch makes the scaled normals of the chunk's
// n extrusions, then n GEMM launches (no gather pass, no gathered copy).  Same draws and the same sums as extrude_once.
int extrude_direct(aog_env* env, bool positive, int n, const double* noise_dev, cudaStream_t st) {
  const aog_config& c = env->cfg;
  const int Np = c.num_pupil_pixels, Ns = c.num_stencil, B = c.num_envs;
  const int flipped = positive ? 1 : 0;
  { int rc = dmma_configure(env); if (rc) return rc; }
  if (n > env->arNZ_cap) {
    int rc = dev_alloc(env, &env->arNZ, (size_t)n * env->chunk * Np);
    if (rc) return rc;
    env->arNZ_cap = n;
  }
  int org = (int)env->cnt.column_origin;
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    dim3 gn(cdiv(cdiv(Np, 4), 64), nB, n);
    k_ar_noise<<<gn, 64, 0, st>>>(noise_dev, env->arNZ, Np, nB, n, e0, env->sqrt_cn2, (long long)n * Np, c.seed,
                                   (unsigned long long)c.env_id_base, (unsigned long long)env->cnt.extrusions);
    AOG_LAUNCH_CHECK();
    org = (int)env->cnt.column_origin;
    for (int i = 0; i < n; ++i) {
      const int phys = positive ? org : (org - 1 + Np) % Np;
      ArDirect dr{};
      dr.nz = env->arNZ + (size_t)i * nB * Np;
      dr.tail = env->t_ar_tail;
      // stencil column x (logical, on the rotated screen when flipped) -> physical column
      dr.pc0 = ((flipped ? Np - 1 : 0) + org) % Np;
      dr.pc1 = ((flipped ? Np - 2 : 1) + org) % Np;
      dr.org = org; dr.Ns = Ns;
      dim3 g2(cdiv(Np, 64), cdiv(nB, AR_TM));
      k_ar_step<true><<<g2, AR_THREADS, AR_SMEM + (Ns - 2 * Np) * (int)sizeof(int), st>>>(nullptr, flipped ? env->t_arW_rev : env->t_arW, env->screens, env->phase_tiles,
                                                      nB, Np, Ns + Np, env->P, e0, phys, flipped,
                                                      1.0 / (c.wavelength_wfs * 3.14159265358979323846), env->phase_tiles_unit, dr);
      AOG_LAUNCH_CHECK();
      org = positive ? (org + 1) % Np : phys;
    }
  }
  env->cnt.column_origin = org;
  env->cnt.extrusions += n;
  return AOG_OK;
}

int evolve_to(aog_env* env, int64_t new_timestep, int64_t old_timestep, const double* noise_dev, cudaStream_t st) {
  if (env->cfg.velocity == 0.0) return AOG_OK;
  const int64_t d = center_px(env, new_timestep) - center_px(env, old_timestep);
  const int Np = env->cfg.num_pupil_pixels;
  const int64_t n = d < 0 ? -d : d;
  if (n == 0) return AOG_OK;
  if (env->ar_direct && n <= 4096) return extrude_direct(env, d > 0, (int)n, noise_dev, st);
  for (int64_t i = 0; i < n; ++i) {
    const double* nz = noise_dev ? noise_dev + (size_t)i * Np : nullptr;
    int rc = extrude_once(env, d > 0, nz, (long long)n * Np, st);
    if (rc) return rc;
  }
  return AOG_OK;
}

// ---- optics chain for one chunk (FP64 path) ---------------------------------------------
int optics_chunk_f64(aog_env* env, int e0, int nB, bool flat_dm, bool with_reward, const aog_outputs& out,
                     cudaStream_t st) {
  const aog_config& c = env->cfg;
  const int Np = c.num_pupil_pixels, Nf = c.num_focal_pixels, n = c.obs_dim, K = c.num_modes, J = c.num_lp_modes;
  const int P = env->P;
  const bool strehl = with_reward && c.rew_type == AOG_REW_STREHL_RATIO;
  constexpr int ET = 4;
  {
    dim3 g(env->strehl_blocks, cdiv(nB, ET));
    k_field_f64<ET><<<g, 128, ET * K * sizeof(double), st>>>(
        env->screens, env->act, env->t_modes, env->t_aperture, env->bufA, env->strehl_part, P, Np, K, e0, nB,
        (int)env->cnt.column_origin, c.wavelength_wfs, c.wavelength_sci, c.amp_fiber, strehl ? 1 : 0,
        flat_dm ? 1 : 0);
    AOG_LAUNCH_CHECK();
  }
  if (env->timing) { AOG_CUDA(cudaEventRecord(env->ev0, st)); }
  {  // T = M1 . E    [Nf x Np] . [Np x Np]
    dim3 g(cdiv(Np, 64), cdiv(Nf, 64), nB);
    k_zgemm<<<g, 256, 0, st>>>(env->t_m1f, env->bufA, env->bufB, Nf, Np, Np, Np, Np, Np, 0, (long long)P,
                               (long long)Nf * Np);
    AOG_LAUNCH_CHECK();
  }
  {  // F = T . M2    [Nf x Np] . [Np x Nf]
    dim3 g(cdiv(Nf, 64), cdiv(Nf, 64), nB);
    k_zgemm<<<g, 256, 0, st>>>(env->bufB, env->t_m2f, env->bufC, Nf, Nf, Np, Np, Nf, Nf, (long long)Nf * Np, 0,
                               (long long)env->NF2);
    AOG_LAUNCH_CHECK();
  }
  if (env->timing) { AOG_CUDA(cudaEventRecord(env->ev1, st)); env->ev_valid = true; }
  const double2 norm = make_double2(c.mft_norm_re, c.mft_norm_im);
  if (with_reward) {
    k_fiber_f64<<<nB, 256, 0, st>>>(env->bufC, env->t_lpw, env->coef, env->NF2, J, (long long)env->NF2, norm);
    AOG_LAUNCH_CHECK();
  }
  {
    dim3 g(cdiv(Np, 8), nB);
    k_obs_rows_f64<<<g, 256, 0, st>>>(env->bufA, env->t_m2o, env->bufR, Np, n, P);
    AOG_LAUNCH_CHECK();
  }
  FinalizeArgs a{};
  a.R = env->bufR; a.m1o = env->t_m1o; a.coef = env->coef; a.lpphase = env->t_lpphase; a.lpgram = env->t_lpgram;
  a.strehl_part = env->strehl_part; a.strehl_blocks = env->strehl_blocks;
  a.Np = Np; a.n = n; a.J = J; a.rew_type = c.rew_type; a.has_thr = c.has_rew_threshold;
  a.compute_reward = with_reward ? 1 : 0;
  a.thr = c.rew_threshold; a.obs_weight = c.obs_weight; a.strehl_scale = c.strehl_scale; a.ssim_peak = c.ssim_ref_peak;
  a.norm = norm;
  const size_t n2 = (size_t)env->n2;
  a.obs16 = out.obs_f16 ? out.obs_f16 + (size_t)e0 * n2 : nullptr;
  a.obs64 = out.obs_f64 ? out.obs_f64 + (size_t)e0 * n2 : nullptr;
  a.reward = out.reward ? out.reward + e0 : nullptr;
  a.power = out.power ? out.power + e0 : nullptr;
  a.strehl = out.strehl ? out.strehl + e0 : nullptr;
  a.ssim = out.ssim ? out.ssim + e0 : nullptr;
  k_finalize<<<nB, 128, 0, st>>>(a);
  AOG_LAUNCH_CHECK();
  return AOG_OK;
}

int optics_all(aog_env* env, bool flat_dm, bool with_reward, const aog_outputs& out, cudaStream_t st) {
  const int B = env->cfg.num_envs;
  if (env->cfg.precision != AOG_PRECISION_F64) return aog_tensor_optics(env, flat_dm, with_reward, out, st);
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    int rc = optics_chunk_f64(env, e0, std::min(env->chunk, B - e0), flat_dm, with_reward, out, st);
    if (rc) return rc;
  }
  return AOG_OK;
}

// device-side outputs of the *_host variants: one allocation [obs64 | reward | power | strehl | ssim | obs16], so that a
// step's results reach the host with ONE device->host copy
int alloc_host_outputs(aog_env* env) {
  const size_t B = env->cfg.num_envs, n2 = env->n2;
  if (env->o_pack) return AOG_OK;
  const size_t bytes = B * n2 * sizeof(double) + 4 * B * sizeof(double) + B * n2 * sizeof(uint16_t);
  int rc;
  if ((rc = dev_alloc(env, &env->o_pack, bytes))) return rc;
  env->o_pack_bytes = bytes;
  AOG_CUDA(cudaMemset(env->o_pack, 0, bytes));
  char* p = env->o_pack;
  env->o_obs64 = (double*)p;   p += B * n2 * sizeof(double);
  env->o_reward = (double*)p;  p += B * sizeof(double);
  env->o_power = (double*)p;   p += B * sizeof(double);
  env->o_strehl = (double*)p;  p += B * sizeof(double);
  env->o_ssim = (double*)p;    p += B * sizeof(double);
  env->o_obs16 = (uint16_t*)p;
  return AOG_OK;
}

// the packed block (already in pinned memory) -> the arrays the caller asked for
void scatter_host_outputs(aog_env* env, const aog_outputs* out) {
  if (!out) return;
  const size_t B = env->cfg.num_envs, n2 = env->n2;
  const char* h = (const char*)env->h_pinned;
  auto take = [&](void* dst, const void* dev, size_t b) {
    if (dst) std::memcpy(dst, h + ((const char*)dev - env->o_pack), b);
  };
  take(out->obs_f64, env->o_obs64, B * n2 * sizeof(double));
  take(out->reward, env->o_reward, B * sizeof(double));
  take(out->power, env->o_power, B * sizeof(double));
  take(out->strehl, env->o_strehl, B * sizeof(double));
  take(out->ssim, env->o_ssim, B * sizeof(double));
  take(out->obs_f16, env->o_obs16, B * n2 * sizeof(uint16_t));
}

// D2H of the outputs through one pinned staging block (one copy), then a stream synchronise.
int copy_outputs_to_host(aog_env* env, const aog_outputs* out, cudaStream_t st) {
  if (!out) { AOG_CUDA(cudaStreamSynchronize(st)); return AOG_OK; }
  int rc = ensure_pinned(env, env->o_pack_bytes);
  if (rc) return rc;
  AOG_CUDA(cudaMemcpyAsync(env->h_pinned, env->o_pack, env->o_pack_bytes, cudaMemcpyDeviceToHost, st));
  AOG_CUDA(cudaStreamSynchronize(st));
  scatter_host_outputs(env, out);
  return AOG_OK;
}

// FP64 scratch (pupil field, stage-1 product, focal field) for handles that did not allocate it at create
int ensure_f64_scratch(aog_env* env) {
  if (env->bufA) return AOG_OK;
  const aog_config& c = env->cfg;
  const size_t ch = env->chunk, P = env->P;
  int rc;
  if ((rc = dev_alloc(env, &env->bufA, ch * P))) return rc;
  if ((rc = dev_alloc(env, &env->bufB, ch * (size_t)c.num_pupil_pixels * std::max(c.num_focal_pixels, c.num_pupil_pixels)))) return rc;
  if ((rc = dev_alloc(env, &env->bufC, ch * std::max<size_t>(env->NF2, P)))) return rc;
  return AOG_OK;
}

aog_outputs device_outputs(aog_env* env) {
  aog_outputs o{};
  o.obs_f16 = env->o_obs16; o.obs_f64 = env->o_obs64; o.reward = env->o_reward; o.power = env->o_power;
  o.strehl = env->o_strehl; o.ssim = env->o_ssim;
  return o;
}

}  // namespace

// ==========================================================================================
extern "C" {

const char* aog_version(void) { return "aogym-b200 0.1 (sm_100a)"; }

const char* aog_last_error(const aog_env* env) { return env ? env->err.c_str() : "null handle"; }

int aog_create(const aog_config* cfg, aog_env** out) {
  if (!cfg || !out) return AOG_ERR_INVALID;
  *out = nullptr;
  aog_env* env = new (std::nothrow) aog_env();
  if (!env) return AOG_ERR_INVALID;
  *out = env;   // returned even on failure so the caller can read aog_last_error, then destroy
  env->cfg = *cfg;
  const aog_config& c = env->cfg;
  if (c.abi_version != AOG_ABI_VERSION) AOG_FAIL(AOG_ERR_INVALID, "abi_version mismatch");
  if (c.num_envs < 1 || c.num_pupil_pixels < 8 || c.num_focal_pixels < 8 || c.num_modes < 1)
    AOG_FAIL(AOG_ERR_INVALID, "bad sizes");
  if (c.obs_dim < 1 || c.obs_dim > AOG_MAX_OBS) AOG_FAIL(AOG_ERR_INVALID, "obs_dim must be in [1, 16]");
  if (c.num_lp_modes < 1 || c.num_lp_modes > AOG_MAX_LP) AOG_FAIL(AOG_ERR_INVALID, "num_lp_modes must be in [1, 8]");
  if (c.rew_type == AOG_REW_SMF_SSIM && c.obs_dim * c.obs_dim < 7)
    AOG_FAIL(AOG_ERR_INVALID, "smf_ssim needs obs_dim^2 >= 7 (SSIM window)");
  int ndev = 0;
  AOG_CUDA(cudaGetDeviceCount(&ndev));
  if (c.device < 0 || c.device >= ndev) AOG_FAIL(AOG_ERR_INVALID, "no such CUDA device");
  AOG_DEVICE(c.device);
  cudaDeviceProp prop;
  AOG_CUDA(cudaGetDeviceProperties(&prop, c.device));
  if (prop.major != 10) AOG_FAIL(AOG_ERR_UNSUPPORTED, "libaogym is built for sm_100a (Blackwell B200) only");
  const int Np = c.num_pupil_pixels, Nf = c.num_focal_pixels, K = c.num_modes, J = c.num_lp_modes, n = c.obs_dim;
  env->P = Np * Np;
  env->NF2 = Nf * Nf;
  env->n2 = n * n;
  const size_t P = env->P, B = c.num_envs;
  int rc;
#define A(expr) if ((rc = (expr))) return rc
  A(dev_alloc(env, &env->t_aperture, P));
  A(dev_alloc(env, &env->t_modes, (size_t)K * P));
  A(dev_alloc(env, &env->t_gram, (size_t)K * K));
  A(dev_alloc(env, &env->t_m1f, (size_t)Nf * Np));
  A(dev_alloc(env, &env->t_m2f, (size_t)Np * Nf));
  A(dev_alloc(env, &env->t_m1o, (size_t)n * Np));
  A(dev_alloc(env, &env->t_m2o, (size_t)Np * n));
  A(dev_alloc(env, &env->t_lpw, (size_t)J * env->NF2));
  A(dev_alloc(env, &env->t_lpphase, (size_t)J));
  A(dev_alloc(env, &env->t_lpgram, (size_t)J * J));
  if (c.num_stencil > 0) {
    A(dev_alloc(env, &env->t_stencil, (size_t)c.num_stencil));
    A(dev_alloc(env, &env->t_arA, (size_t)Np * c.num_stencil));
    A(dev_alloc(env, &env->t_arB, (size_t)Np * Np));
    A(dev_alloc(env, &env->t_arW, (size_t)(c.num_stencil + Np) * Np));
    A(dev_alloc(env, &env->t_arW_rev, (size_t)(c.num_stencil + Np) * Np));
  }
  if (c.num_screen_fine > 0) {
    const size_t N2 = c.num_screen_fine;
    A(dev_alloc(env, &env->t_scrC1, P));
    A(dev_alloc(env, &env->t_scrW1, P));
    A(dev_alloc(env, &env->t_scrW1T, P));
    A(dev_alloc(env, &env->t_scrC2, N2 * N2));
    A(dev_alloc(env, &env->t_scrW2, (size_t)Np * N2));
    A(dev_alloc(env, &env->t_scrW2T, (size_t)Np * N2));
  }
  A(dev_alloc(env, &env->screens, B * P));
  AOG_CUDA(cudaMemset(env->screens, 0, B * P * sizeof(double)));
  A(dev_alloc(env, &env->act, B * K));
  AOG_CUDA(cudaMemset(env->act, 0, B * K * sizeof(double)));
  A(dev_alloc(env, (double**)&env->act_in, B * K));
  // every env starts at the configured strength (aog_set_turbulence changes it per env)
  env->sqrt_cn2_host.assign(B, c.sqrt_cn2);
  A(dev_alloc(env, &env->sqrt_cn2, 2 * B));
  AOG_CUDA(cudaMemcpy(env->sqrt_cn2, env->sqrt_cn2_host.data(), B * sizeof(double), cudaMemcpyHostToDevice));
  env->chunk = (int)std::min<size_t>(B, 4096);
  env->strehl_blocks = cdiv(env->P, 128);
  const size_t ch = env->chunk;
  if (c.precision == AOG_PRECISION_F64 || c.num_screen_fine > 0) {
    A(dev_alloc(env, &env->bufA, ch * P));
    A(dev_alloc(env, &env->bufB, ch * (size_t)Np * std::max(Nf, Np)));
    A(dev_alloc(env, &env->bufC, ch * std::max<size_t>(env->NF2, P)));
  }
  A(dev_alloc(env, &env->bufR, ch * (size_t)Np * n));
  A(dev_alloc(env, &env->coef, ch * (size_t)J));
  A(dev_alloc(env, &env->strehl_part, ch * (size_t)env->strehl_blocks));
  if (c.num_stencil > 0) {
    A(dev_alloc(env, &env->arZ, ch * (size_t)(c.num_stencil + Np)));
  }
  A(alloc_host_outputs(env));
  if (c.precision != AOG_PRECISION_F64) A(aog_tensor_create(env));
#undef A
  AOG_CUDA(cudaStreamCreate(&env->own_stream));   // blocking: ordered with the default stream
  {
    // highest priority: its (few, compute-bound) blocks are placed as soon as an SM has room, next to the HBM-bound
    // blocks of the kernels they overlap with
    int lo = 0, hi = 0;
    AOG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    AOG_CUDA(cudaStreamCreateWithPriority(&env->side_stream, cudaStreamNonBlocking, hi));
  }
  AOG_CUDA(cudaEventCreateWithFlags(&env->ev_sh_phase, cudaEventDisableTiming));
  AOG_CUDA(cudaEventCreateWithFlags(&env->ev_ext_done, cudaEventDisableTiming));
  AOG_CUDA(cudaEventCreate(&env->ev0));
  AOG_CUDA(cudaEventCreate(&env->ev1));
  AOG_CUDA(cudaEventCreate(&env->evf));
  AOG_CUDA(cudaEventCreate(&env->evm));
  for (auto& e : env->tev) AOG_CUDA(cudaEventCreate(&e));
  return AOG_OK;
}

void aog_destroy(aog_env* env) {
  if (!env) return;
  DeviceGuard guard(env->cfg.device);
  cudaDeviceSynchronize();
  aog_tensor_destroy(env);
  void* ptrs[] = {env->t_aperture, env->t_modes, env->t_gram, env->t_m1f, env->t_m2f, env->t_m1o, env->t_m2o,
                  env->t_lpw, env->t_lpphase, env->t_lpgram, env->t_stencil, env->t_stencil_perm, env->t_arA, env->t_arB, env->t_arW,
                  env->t_arW_rev, env->t_ar_tail, env->arNZ, env->t_scr_sh, env->t_scr_tw, env->t_scrC1, env->t_scrW1, env->t_scrW1T, env->t_scrC2, env->t_scrW2, env->t_scrW2T,
                  env->screens, env->act, env->sqrt_cn2, env->bufA, env->bufB, env->bufC, env->bufR, env->coef,
                  env->strehl_part, env->arZ, env->act_in, env->noise_in, env->o_pack,
                  env->t_sh_mla, env->t_sh_C, env->t_sh_CT,
                  env->t_sh_off, env->t_sh_pix, env->t_sh_px, env->t_sh_py, env->t_sh_offset, env->t_sh_recon,
                  env->t_sh_act0, env->act_sh, env->o_action, env->sh_noisy_in, env->t_sh_Cf[0], env->t_sh_Cf[1],
                  env->t_sh_Cf[2], env->t_sh_Cf[3], env->t_scrWst[0], env->t_scrWst[1], env->t_scrWrT[0], env->t_scrWrT[1],
                  env->t_scrWiT[0], env->t_scrWiT[1]};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (env->h_pinned) cudaFreeHost(env->h_pinned);
  if (env->h_act) cudaFreeHost(env->h_act);
  if (env->step_graph) cudaGraphExecDestroy(env->step_graph);
  if (env->own_stream) cudaStreamDestroy(env->own_stream);
  if (env->side_stream) cudaStreamDestroy(env->side_stream);
  if (env->ev_sh_phase) cudaEventDestroy(env->ev_sh_phase);
  if (env->ev_ext_done) cudaEventDestroy(env->ev_ext_done);
  if (env->ev0) cudaEventDestroy(env->ev0);
  if (env->ev1) cudaEventDestroy(env->ev1);
  if (env->evf) cudaEventDestroy(env->evf);
  if (env->evm) cudaEventDestroy(env->evm);
  for (auto& e : env->tev)
    if (e) cudaEventDestroy(e);
  delete env;
}

int aog_set_table(aog_env* env, int which, const void* host, size_t count) {
  if (!env || !host) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  AOG_DEVICE(c.device);
  const size_t Np = c.num_pupil_pixels, Nf = c.num_focal_pixels, K = c.num_modes, J = c.num_lp_modes, n = c.obs_dim;
  const size_t P = env->P, Ns = c.num_stencil, N2 = c.num_screen_fine;
  void* dst = nullptr;
  size_t want = 0, esz = sizeof(double);
  switch (which) {
    case AOG_TABLE_APERTURE: dst = env->t_aperture; want = P; break;
    case AOG_TABLE_DM_MODES: dst = env->t_modes; want = K * P; break;
    case AOG_TABLE_DM_GRAM: dst = env->t_gram; want = K * K; break;
    case AOG_TABLE_MFT_FIB_1: dst = env->t_m1f; want = Nf * Np; esz = sizeof(double2); break;
    case AOG_TABLE_MFT_FIB_2: dst = env->t_m2f; want = Np * Nf; esz = sizeof(double2); break;
    case AOG_TABLE_MFT_OBS_1: dst = env->t_m1o; want = n * Np; esz = sizeof(double2); break;
    case AOG_TABLE_MFT_OBS_2: dst = env->t_m2o; want = Np * n; esz = sizeof(double2); break;
    case AOG_TABLE_LP_MODES_W: dst = env->t_lpw; want = J * env->NF2; break;
    case AOG_TABLE_LP_PHASE: dst = env->t_lpphase; want = J; esz = sizeof(double2); break;
    case AOG_TABLE_LP_GRAM: dst = env->t_lpgram; want = J * J; break;
    case AOG_TABLE_AR_STENCIL: dst = env->t_stencil; want = Ns; esz = sizeof(int32_t); break;
    case AOG_TABLE_AR_A: dst = env->t_arA; want = Np * Ns; break;
    case AOG_TABLE_AR_B: dst = env->t_arB; want = Np * Np; break;
    case AOG_TABLE_SCR_C1: dst = env->t_scrC1; want = P; break;
    case AOG_TABLE_SCR_W1: dst = env->t_scrW1; want = P; esz = sizeof(double2); break;
    case AOG_TABLE_SCR_C2: dst = env->t_scrC2; want = N2 * N2; break;
    case AOG_TABLE_SCR_W2: dst = env->t_scrW2; want = Np * N2; esz = sizeof(double2); break;
    case AOG_TABLE_SH_MLA_PHASE: dst = env->t_sh_mla; want = P; break;
    case AOG_TABLE_SH_FRESNEL: dst = env->t_sh_C; want = P; esz = sizeof(double2); break;
    case AOG_TABLE_SH_PIX_OFFSETS: dst = env->t_sh_off; want = (size_t)env->sh_num_sub + 1; esz = sizeof(int32_t); break;
    case AOG_TABLE_SH_PIX_INDEX: dst = env->t_sh_pix; want = (size_t)env->sh_num_pix; esz = sizeof(int32_t); break;
    case AOG_TABLE_SH_PIX_X: dst = env->t_sh_px; want = (size_t)env->sh_num_pix; break;
    case AOG_TABLE_SH_PIX_Y: dst = env->t_sh_py; want = (size_t)env->sh_num_pix; break;
    case AOG_TABLE_SH_OFFSET: dst = env->t_sh_offset; want = 2 * (size_t)env->sh_num_sub; break;
    case AOG_TABLE_SH_RECON: dst = env->t_sh_recon; want = K * 2 * (size_t)env->sh_num_sub; break;
    case AOG_TABLE_SH_ACT0: dst = env->t_sh_act0; want = K; break;
    default: AOG_FAIL(AOG_ERR_INVALID, "unknown table id");
  }
  if (!dst || want == 0) AOG_FAIL(AOG_ERR_INVALID, "table not configured for this handle");
  if (count != want)
    AOG_FAIL(AOG_ERR_INVALID, "table " + std::to_string(which) + ": expected " + std::to_string(want) +
                                  " elements, got " + std::to_string(count));
  if (which == AOG_TABLE_AR_STENCIL) {
    // gather order = by column, then row: the first stencil columns become contiguous runs of the column-major
    // screens (coalesced gather); the rows of W follow the same permutation (k_build_arW)
    const int32_t* st = static_cast<const int32_t*>(host);
    std::vector<int> perm(Ns), sorted(Ns);
    for (size_t j = 0; j < Ns; ++j) perm[j] = (int)j;
    std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) {
      const long long ka = (long long)(st[a] % (int)Np) * (long long)Np + st[a] / (int)Np;
      const long long kb = (long long)(st[b] % (int)Np) * (long long)Np + st[b] / (int)Np;
      return ka < kb;
    });
    for (size_t j = 0; j < Ns; ++j) sorted[j] = st[perm[j]];
    int rc = dev_alloc(env, &env->t_stencil_perm, Ns);
    if (rc) return rc;
    AOG_CUDA(cudaMemcpy(env->t_stencil_perm, perm.data(), Ns * sizeof(int), cudaMemcpyHostToDevice));
    AOG_CUDA(cudaMemcpy(dst, sorted.data(), Ns * sizeof(int), cudaMemcpyHostToDevice));
    // hcipy's stencil (two full columns + one pixel per row further back) lets k_ar_step read the screens in place
    bool direct = Np % 2 == 0 && Ns > 2 * Np && Ns - 2 * Np <= 4096 && getenv("AOG_AR_GATHER") == nullptr;
    for (size_t k = 0; direct && k < 2 * Np; ++k) direct = sorted[k] == (int)((k % Np) * Np + k / Np);
    std::vector<int> tail(Ns > 2 * Np ? Ns - 2 * Np : 0);
    for (size_t k = 2 * Np; direct && k < Ns; ++k) {
      const int x = sorted[k] % (int)Np, y = sorted[k] / (int)Np;
      direct = x >= 2 && x <= (int)Np - 2;            // never the column an extrusion overwrites (logical Np - 1)
      tail[k - 2 * Np] = x | (y << 16);
    }
    env->ar_direct = direct;
    if (direct) {
      rc = dev_alloc(env, &env->t_ar_tail, tail.size());
      if (rc) return rc;
      AOG_CUDA(cudaMemcpy(env->t_ar_tail, tail.data(), tail.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
  } else {
    AOG_CUDA(cudaMemcpy(dst, host, want * esz, cudaMemcpyHostToDevice));
  }
  env->have[which] = true;
  if (env->step_graph) { cudaGraphExecDestroy(env->step_graph); env->step_graph = nullptr; }   // captured launches hold table-derived arguments
  if ((which == AOG_TABLE_AR_A || which == AOG_TABLE_AR_B || which == AOG_TABLE_AR_STENCIL) && env->have[AOG_TABLE_AR_A] &&
      env->have[AOG_TABLE_AR_B] && env->have[AOG_TABLE_AR_STENCIL]) {
    const int tot = (int)((Ns + Np) * Np);
    k_build_arW<<<cdiv(tot, 256), 256>>>(env->t_arA, env->t_arB, env->t_stencil_perm, env->t_arW, (int)Np, (int)Ns, 0);
    AOG_LAUNCH_CHECK();
    k_build_arW<<<cdiv(tot, 256), 256>>>(env->t_arA, env->t_arB, env->t_stencil_perm, env->t_arW_rev, (int)Np, (int)Ns, 1);
    AOG_LAUNCH_CHECK();
  }
  if (which == AOG_TABLE_SCR_W1) {
    k_transpose_z<<<cdiv((int)P, 256), 256>>>(env->t_scrW1, env->t_scrW1T, (int)Np, (int)Np);
    AOG_LAUNCH_CHECK();
  }
  if (which == AOG_TABLE_SCR_W1) {
    // a shifted DFT matrix of the reference size?  W1[x][k] = W1[0][k] exp(2 pi i x k / N)  ->  FFT synthesis
    const double* m = static_cast<const double*>(host);
    const size_t N = Np;
    bool fft = N == 240 && getenv("AOG_SCR_GEMM") == nullptr && getenv("AOG_SCR_COMPLEX") == nullptr;
    std::vector<double> tw(2 * 240);
    for (int j = 0; j < 240; ++j) {
      tw[2 * j] = std::cos(2.0 * 3.14159265358979323846 * j / 240.0);
      tw[2 * j + 1] = std::sin(2.0 * 3.14159265358979323846 * j / 240.0);
    }
    double res = 0.0;
    for (size_t x = 0; fft && x < N; ++x)
      for (size_t k = 0; k < N; ++k) {
        const size_t j = (x * k) % N;
        const double sr = m[2 * k], si = m[2 * k + 1];
        const double er = sr * tw[2 * j] - si * tw[2 * j + 1], ei = sr * tw[2 * j + 1] + si * tw[2 * j];
        res = std::max(res, std::max(std::fabs(m[2 * (x * N + k)] - er), std::fabs(m[2 * (x * N + k) + 1] - ei)));
      }
    env->scr_fft = fft && res <= 1e-11;
    if (env->scr_fft) {
      int rc;
      if ((rc = dev_alloc(env, &env->t_scr_sh, N))) return rc;
      if ((rc = dev_alloc(env, &env->t_scr_tw, (size_t)240))) return rc;
      AOG_CUDA(cudaMemcpy(env->t_scr_sh, m, N * sizeof(double2), cudaMemcpyHostToDevice));       // row x = 0
      AOG_CUDA(cudaMemcpy(env->t_scr_tw, tw.data(), 240 * sizeof(double2), cudaMemcpyHostToDevice));
    }
  }
  if (which == AOG_TABLE_SCR_W1 || which == AOG_TABLE_SCR_W2) {
    // conjugate-paired rows -> real-arithmetic synthesis tables (common.cuh: t_scrWst)
    const int sidx = which == AOG_TABLE_SCR_W1 ? 0 : 1;
    const size_t N = Np, Nh = Np / 2, Nk = sidx == 0 ? Np : N2;
    const double* m = static_cast<const double*>(host);      // [N][Nk] complex
    double mx = 0.0, res = 0.0;
    for (size_t x = 0; x < N; ++x)
      for (size_t k = 0; k < Nk; ++k) {
        const double* a = &m[2 * (x * Nk + k)];
        const double* b = &m[2 * ((N - 1 - x) * Nk + k)];
        mx = std::max(mx, std::max(std::fabs(a[0]), std::fabs(a[1])));
        res = std::max(res, std::max(std::fabs(a[0] - b[0]), std::fabs(a[1] + b[1])));
      }
    env->scr_sym[sidx] = N % 2 == 0 && Nk % 2 == 0 && res <= 1e-12 * mx && getenv("AOG_SCR_COMPLEX") == nullptr;
    if (env->scr_sym[sidx]) {
      std::vector<double> wst(N * Nk), wrT(Nk * Nh), wiT(Nk * Nh);
      for (size_t x = 0; x < Nh; ++x)
        for (size_t k = 0; k < Nk; ++k) {
          const double re = m[2 * (x * Nk + k)], im = m[2 * (x * Nk + k) + 1];
          wst[x * Nk + k] = re;
          wst[(Nh + x) * Nk + k] = im;
          wrT[k * Nh + x] = re;
          wiT[k * Nh + x] = im;
        }
      int rc;
      if ((rc = dev_alloc(env, &env->t_scrWst[sidx], N * Nk))) return rc;
      if ((rc = dev_alloc(env, &env->t_scrWrT[sidx], Nk * Nh))) return rc;
      if ((rc = dev_alloc(env, &env->t_scrWiT[sidx], Nk * Nh))) return rc;
      AOG_CUDA(cudaMemcpy(env->t_scrWst[sidx], wst.data(), wst.size() * sizeof(double), cudaMemcpyHostToDevice));
      AOG_CUDA(cudaMemcpy(env->t_scrWrT[sidx], wrT.data(), wrT.size() * sizeof(double), cudaMemcpyHostToDevice));
      AOG_CUDA(cudaMemcpy(env->t_scrWiT[sidx], wiT.data(), wiT.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
  }
  if (which == AOG_TABLE_SH_FRESNEL) {
    k_transpose_z<<<cdiv((int)P, 256), 256>>>(env->t_sh_C, env->t_sh_CT, (int)Np, (int)Np);
    AOG_LAUNCH_CHECK();
    // centrosymmetric operator -> parity-folded tables (common.cuh: t_sh_Cf)
    const double* m = static_cast<const double*>(host);
    const size_t N = Np, Nh = Np / 2;
    double mx = 0.0, res = 0.0;
    for (size_t i = 0; i < N; ++i)
      for (size_t j = 0; j < N; ++j) {
        const double* a = &m[2 * (i * N + j)];
        const double* b = &m[2 * ((N - 1 - i) * N + (N - 1 - j))];
        mx = std::max(mx, std::max(std::fabs(a[0]), std::fabs(a[1])));
        res = std::max(res, std::max(std::fabs(a[0] - b[0]), std::fabs(a[1] - b[1])));
      }
    env->sh_fold = (N % 2 == 0) && res <= 1e-13 * mx && getenv("AOG_SH_NO_FOLD") == nullptr;
    if (env->sh_fold) {
      std::vector<double> t(4 * 2 * Nh * Nh);
      for (size_t i = 0; i < Nh; ++i)
        for (size_t j = 0; j < Nh; ++j) {
          const double* a = &m[2 * (i * N + j)];
          const double* b = &m[2 * (i * N + (N - 1 - j))];
          for (int c = 0; c < 2; ++c) {
            const double ce = 0.5 * (a[c] + b[c]), co = 0.5 * (a[c] - b[c]);
            t[0 * 2 * Nh * Nh + 2 * (i * Nh + j) + c] = ce;
            t[1 * 2 * Nh * Nh + 2 * (i * Nh + j) + c] = co;
            t[2 * 2 * Nh * Nh + 2 * (j * Nh + i) + c] = ce;
            t[3 * 2 * Nh * Nh + 2 * (j * Nh + i) + c] = co;
          }
        }
      for (int k = 0; k < 4; ++k) {
        int rc = dev_alloc(env, &env->t_sh_Cf[k], Nh * Nh);
        if (rc) return rc;
        AOG_CUDA(cudaMemcpy(env->t_sh_Cf[k], &t[(size_t)k * 2 * Nh * Nh], Nh * Nh * sizeof(double2), cudaMemcpyHostToDevice));
      }
    }
  }
  if (which == AOG_TABLE_SH_ACT0) {   // every env's SH mirror starts from the same actuators (AO_env.py:431-447)
    k_broadcast_rows<<<cdiv((int)K * c.num_envs, 256), 256>>>(env->t_sh_act0, env->act_sh, (int)K, c.num_envs);
    AOG_LAUNCH_CHECK();
  }
  if (which == AOG_TABLE_SCR_W2) {
    k_transpose_z<<<cdiv((int)(Np * N2), 256), 256>>>(env->t_scrW2, env->t_scrW2T, (int)Np, (int)N2);
    AOG_LAUNCH_CHECK();
  }
  if (c.precision != AOG_PRECISION_F64) {
    int rc = aog_tensor_table_updated(env, which, host);
    if (rc) return rc;
  }
  AOG_CUDA(cudaDeviceSynchronize());
  return AOG_OK;
}

int aog_set_screens(aog_env* env, const void* src, int dtype, int src_on_device, int first_env, int count) {
  if (!env || !src) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (first_env < 0 || count < 1 || first_env + count > c.num_envs) AOG_FAIL(AOG_ERR_INVALID, "env range");
  AOG_DEVICE(c.device);
  const size_t nel = (size_t)count * env->P;
  double* dst = env->screens + (size_t)first_env * env->P;
  if (env->cnt.column_origin != 0) AOG_FAIL(AOG_ERR_STATE, "set_screens after extrusions: reset counters first");
  if (dtype != AOG_DTYPE_F64 && dtype != AOG_DTYPE_F32) AOG_FAIL(AOG_ERR_INVALID, "dtype");
  {
    // the caller's screens are [y][x] (hcipy Field order); the device keeps them column-major
    const size_t esz = dtype == AOG_DTYPE_F64 ? sizeof(double) : sizeof(float);
    const void* s = src;
    void* tmp = nullptr;
    if (!src_on_device) {
      AOG_CUDA(cudaMalloc(&tmp, nel * esz));
      cudaError_t e = cudaMemcpy(tmp, src, nel * esz, cudaMemcpyHostToDevice);
      if (e != cudaSuccess) { cudaFree(tmp); env->err = cudaGetErrorString(e); return AOG_ERR_CUDA; }
      s = tmp;
    }
    const unsigned grid = (unsigned)((nel + 255) / 256);
    if (dtype == AOG_DTYPE_F64) k_screens_in<double><<<grid, 256>>>((const double*)s, dst, c.num_pupil_pixels, nel);
    else k_screens_in<float><<<grid, 256>>>((const float*)s, dst, c.num_pupil_pixels, nel);
    env->launches++;
    cudaError_t e = cudaDeviceSynchronize();
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) { env->err = cudaGetErrorString(e); return AOG_ERR_CUDA; }
  }
  if (c.precision != AOG_PRECISION_F64) return aog_tensor_screens_updated(env);
  return AOG_OK;
}

int aog_get_screens(aog_env* env, double* host_out, int first_env, int count) {
  if (!env || !host_out) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (first_env < 0 || count < 1 || first_env + count > c.num_envs) AOG_FAIL(AOG_ERR_INVALID, "env range");
  AOG_DEVICE(c.device);
  AOG_CUDA(cudaDeviceSynchronize());
  const int Np = c.num_pupil_pixels, org = (int)env->cnt.column_origin;
  std::vector<double> tmp((size_t)count * env->P);
  AOG_CUDA(cudaMemcpy(tmp.data(), env->screens + (size_t)first_env * env->P, tmp.size() * sizeof(double),
                      cudaMemcpyDeviceToHost));
  for (int b = 0; b < count; ++b)
    for (int y = 0; y < Np; ++y)
      for (int x = 0; x < Np; ++x)
        host_out[(size_t)b * env->P + (size_t)y * Np + x] = tmp[(size_t)b * env->P + (size_t)((x + org) % Np) * Np + y];
  return AOG_OK;
}

int aog_generate_screens(aog_env* env, void* stream) {
  if (!env) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (c.num_screen_fine <= 0 || !env->have[AOG_TABLE_SCR_C1] || !env->have[AOG_TABLE_SCR_W1] ||
      !env->have[AOG_TABLE_SCR_C2] || !env->have[AOG_TABLE_SCR_W2])
    AOG_FAIL(AOG_ERR_STATE, "screen synthesis tables not set");
  AOG_DEVICE(c.device);
  cudaStream_t st = (cudaStream_t)stream;
  const int Np = c.num_pupil_pixels, N2 = c.num_screen_fine, P = env->P, B = c.num_envs;
  // independent Philox domain from the extrusion noise: offset the seed
  const unsigned long long seed = c.seed ^ 0x9E3779B97F4A7C15ull;
  const unsigned long long per = (unsigned long long)P + (unsigned long long)N2 * N2;
  const unsigned long long base = (unsigned long long)(env->screen_draws++) * per;
  const long long sB = (long long)Np * std::max(c.num_focal_pixels, Np);
  const long long sC = (long long)std::max<size_t>(env->NF2, P);
  // real-arithmetic form on the FP64 tensor cores (common.cuh: t_scrWst), one scale at a time:
  //   out1 = [Re W_top ; Im W_top] . [Xr | Xi]   (N x 2 Nk)  ->  U = rows < N/2, V = rows >= N/2
  //   P1 = Ur WrT, P2 = Vi WrT, P3 = Ui WiT, P4 = Vr WiT   (N/2 x N/2 each)  ->  k_scr_combine4
  const bool fft_form = env->scr_fft && Np == 240 && env->scr_sym[0] && env->scr_sym[1] && N2 % 2 == 0;
  bool tiles_done = fft_form && env->phase_tiles != nullptr;       // k_scr_fft_cols refreshes the phase tiles itself
  auto synth_real = [&](int sidx, int Nk, const double* Ctab, unsigned long long draw_base, int e0, int nB,
                        int accumulate) -> int {
    const int Nh = Np / 2, Q = Nh * Nh;
    double* X = reinterpret_cast<double*>(env->bufA);
    double* O = reinterpret_cast<double*>(env->bufB);
    double* Pq = reinterpret_cast<double*>(env->bufC);
    const long long sX = 2LL * P, sO = 2 * sB, sP = 2 * sC;
    { int rc = dmma_configure(env); if (rc) return rc; }
    if (sidx == 0 && fft_form) {
      // the fine scale is a 240 x 240 inverse DFT: rows (normals drawn in the kernel), then columns straight into
      // the screens, on top of the coarse scale, with the phase tiles of the tensor / fused paths (fft240.cuh)
      double2* T = env->bufB;
      k_scr_fft_rows<<<dim3(240 / FFT_LINES, nB), FFT_THREADS, FFT_SMEM, st>>>(Ctab, env->t_scr_sh, env->t_scr_tw, T, sB, e0, seed,
                                                                       (unsigned long long)c.env_id_base, draw_base);
      AOG_LAUNCH_CHECK();
      k_scr_fft_cols<<<dim3(240 / FFT_LINES, nB), FFT_THREADS, FFT_SMEM, st>>>(T, sB, env->t_scr_tw, env->screens, P, e0, env->sqrt_cn2, accumulate,
                                                                       nullptr, 0.0, 0.0);
      AOG_LAUNCH_CHECK();
      return AOG_OK;
    }
    k_scr_noise_planes<<<dim3(cdiv(Nk * Nk / 2, 256), nB), 256, 0, st>>>(Ctab, X, Nk, sX, e0, seed,
                                                                          (unsigned long long)c.env_id_base, draw_base);
    AOG_LAUNCH_CHECK();
    k_dgemm_mma<<<dim3(cdiv(2 * Nk, 64), cdiv(Np, 128), nB), 256, DmmaCfg<1>::SMEM, st>>>(env->t_scrWst[sidx], X, O, Np, 2 * Nk, Nk, Nk,
                                                                           2 * Nk, 2 * Nk, 0, sX, sO);
    AOG_LAUNCH_CHECK();
    const double* Aop[4] = {O, O + (size_t)Nh * 2 * Nk + Nk, O + Nk, O + (size_t)Nh * 2 * Nk};      // Ur, Vi, Ui, Vr
    const double* Bop[4] = {env->t_scrWrT[sidx], env->t_scrWrT[sidx], env->t_scrWiT[sidx], env->t_scrWiT[sidx]};
    for (int q = 0; q < 4; ++q) {
      k_dgemm_mma<<<dim3(cdiv(Nh, 64), cdiv(Nh, 128), nB), 256, DmmaCfg<1>::SMEM, st>>>(Aop[q], Bop[q], Pq + (size_t)q * Q, Nh, Nh, Nk,
                                                                         2 * Nk, Nh, Nh, sO, 0, sP);
      AOG_LAUNCH_CHECK();
    }
    // with the FFT form this is the last writer of the screens: it also refreshes the phase tiles
    const bool wt = fft_form && accumulate && env->phase_tiles != nullptr;
    k_scr_combine4<<<dim3(cdiv(Q, 256), nB), 256, 0, st>>>(env->screens, Pq, Np, sP, e0, env->sqrt_cn2, accumulate,
                                                           wt ? env->phase_tiles : nullptr,
                                                           1.0 / (c.wavelength_wfs * 3.14159265358979323846), env->phase_tiles_unit);
    AOG_LAUNCH_CHECK();
    return AOG_OK;
  };
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    if (env->scr_sym[0] && env->scr_sym[1]) {
      int rc = synth_real(0, Np, env->t_scrC1, base, e0, nB, 0);
      if (rc) return rc;
      rc = synth_real(1, N2, env->t_scrC2, base + P, e0, nB, 1);
      if (rc) return rc;
      continue;
    }
    tiles_done = false;
    // scale 1: X1 [Np x Np] -> W1 X1 W1^T
    k_scr_noise<<<dim3(cdiv(P / 2, 256), nB), 256, 0, st>>>(env->t_scrC1, env->bufA, P, (long long)P, e0, seed,
                                                        (unsigned long long)c.env_id_base, base);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->t_scrW1, env->bufA, env->bufB, Np, Np, Np, Np,
                                                                   Np, Np, 0, (long long)P, sB);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->bufB, env->t_scrW1T, env->bufC, Np, Np, Np, Np,
                                                                   Np, Np, sB, 0, sC);
    AOG_LAUNCH_CHECK();
    k_scr_combine<<<dim3(cdiv(P, 256), nB), 256, 0, st>>>(env->screens, env->bufC, P, sC, e0, env->sqrt_cn2, 0);
    AOG_LAUNCH_CHECK();
    // scale 2: X2 [N2 x N2] -> W2 X2 W2^T
    k_scr_noise<<<dim3(cdiv(N2 * N2 / 2, 256), nB), 256, 0, st>>>(env->t_scrC2, env->bufA, N2 * N2, (long long)P, e0, seed,
                                                              (unsigned long long)c.env_id_base, base + P);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(N2, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->t_scrW2, env->bufA, env->bufB, Np, N2, N2, N2,
                                                                   N2, N2, 0, (long long)P, sB);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->bufB, env->t_scrW2T, env->bufC, Np, Np, N2, N2,
                                                                   Np, Np, sB, 0, sC);
    AOG_LAUNCH_CHECK();
    k_scr_combine<<<dim3(cdiv(P, 256), nB), 256, 0, st>>>(env->screens, env->bufC, P, sC, e0, env->sqrt_cn2, 1);
    AOG_LAUNCH_CHECK();
  }
  env->cnt.column_origin = 0;
  if (c.precision != AOG_PRECISION_F64 && !tiles_done) return aog_tensor_screens_updated(env);
  return AOG_OK;
}

int aog_set_turbulence(aog_env* env, const double* sqrt_cn2_host, int rescale, void* stream) {
  if (!env || !sqrt_cn2_host) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  const int B = c.num_envs;
  for (int b = 0; b < B; ++b)
    if (!std::isfinite(sqrt_cn2_host[b]) || !(sqrt_cn2_host[b] > 0.0))
      AOG_FAIL(AOG_ERR_INVALID, "sqrt_cn2 of env " + std::to_string(b) + " is not finite and positive");
  AOG_DEVICE(c.device);
  cudaStream_t st = (cudaStream_t)stream;
  // [new values | new / old]: one upload (pageable source: staged before cudaMemcpyAsync returns)
  std::vector<double> h(rescale ? 2 * (size_t)B : (size_t)B);
  for (int b = 0; b < B; ++b) {
    h[b] = sqrt_cn2_host[b];
    if (rescale) h[B + b] = sqrt_cn2_host[b] / env->sqrt_cn2_host[b];
  }
  AOG_CUDA(cudaMemcpyAsync(env->sqrt_cn2, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  env->sqrt_cn2_host.assign(sqrt_cn2_host, sqrt_cn2_host + B);
  if (!rescale) return AOG_OK;
  // the screens are a linear function of sqrt(Cn^2) (synthesis and AR extrusion alike): the same realisation at the new
  // strength.  Elementwise, so the ring origin does not matter.
  const double* factor = env->sqrt_cn2 + B;
  if (env->phase_tiles) return aog_tensor_rescale_screens(env, factor, st);
  const size_t total = (size_t)B * env->P;
  k_scale_screens<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(env->screens, factor, env->P, total);
  AOG_LAUNCH_CHECK();
  return AOG_OK;
}

int aog_next_extrusions(const aog_env* env) {
  if (!env) return AOG_ERR_INVALID;
  if (env->cfg.velocity == 0.0) return 0;
  const int64_t d = center_px(env, env->cnt.timestep + 1) - center_px(env, env->cnt.timestep);
  return (int)(d < 0 ? -d : d);
}

int aog_reset(aog_env* env, const aog_outputs* out_dev, void* stream) {
  if (!env) return AOG_ERR_INVALID;
  if (!tables_ready(env)) return AOG_ERR_STATE;
  const aog_config& c = env->cfg;
  AOG_DEVICE(c.device);
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  // AO_env.py:76-77 -- semi_dynamic draws a fresh screen per episode
  if (c.atm_type == AOG_ATM_SEMI_DYNAMIC && c.num_screen_fine > 0)
    if ((rc = aog_generate_screens(env, st))) return rc;
  // AO_env.py:79-80
  if (c.flat_mirror_start) AOG_CUDA(cudaMemsetAsync(env->act, 0, (size_t)c.num_envs * c.num_modes * sizeof(double), st));
  env->cnt.timestep_render = 0;           // AO_env.py:83
  // AO_env.py:84: layer.t = timestep * delta_t -- same time as the last step: no extrusion
  aog_outputs o{};
  if (out_dev) o = *out_dev;
  o.reward = nullptr; o.power = nullptr; o.strehl = nullptr; o.ssim = nullptr;
  return optics_all(env, false, false, o, st);
}

int aog_reset_host(aog_env* env, const aog_outputs* out_host) {
  if (!env) return AOG_ERR_INVALID;
  aog_outputs d = device_outputs(env);
  int rc = aog_reset(env, &d, env->own_stream);
  if (rc) return rc;
  aog_outputs h{};
  if (out_host) { h.obs_f16 = out_host->obs_f16; h.obs_f64 = out_host->obs_f64; }
  return copy_outputs_to_host(env, &h, env->own_stream);
}

int aog_step(aog_env* env, const void* actions_dev, int act_dtype, const double* noise_dev,
             const aog_outputs* out_dev, int32_t* done_out, void* stream) {
  if (!env || !actions_dev) return AOG_ERR_INVALID;
  if (!tables_ready(env)) return AOG_ERR_STATE;
  const aog_config& c = env->cfg;
  AOG_DEVICE(c.device);
  cudaStream_t st = (cudaStream_t)stream;
  const int B = c.num_envs, K = c.num_modes;
  // AO_env.py:115-120
  const size_t shm = (size_t)(K + 32) * sizeof(double);
  const double target = 0.1 * c.wavelength_sci;
  if (act_dtype != AOG_DTYPE_F32 && act_dtype != AOG_DTYPE_F64) AOG_FAIL(AOG_ERR_INVALID, "act_dtype");
  int arc = AOG_ERR_UNSUPPORTED;
  if (c.precision != AOG_PRECISION_F64) {
    arc = aog_tensor_actuators(env, actions_dev, act_dtype, st);
    if (arc != AOG_OK && arc != AOG_ERR_UNSUPPORTED) return arc;
  }
  if (arc != AOG_OK) {
    if (act_dtype == AOG_DTYPE_F32)
      k_actuators<float><<<B, 128, shm, st>>>((const float*)actions_dev, env->t_gram, env->act, K, c.sh_operation, target);
    else
      k_actuators<double><<<B, 128, shm, st>>>((const double*)actions_dev, env->t_gram, env->act, K, c.sh_operation, target);
    AOG_LAUNCH_CHECK();
  }
  // AO_env.py:123-125
  const int64_t old_t = env->cnt.timestep;
  env->cnt.timestep += 1;
  env->cnt.timestep_render += 1;
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[0], st));
  const int64_t ext_before = env->cnt.extrusions;
  int rc;
  if (env->sh_phase_pending && env->sh_phase_stream == st && c.velocity != 0.0 && !env->timing) {
    // SH_step's phase kernel was the last reader of the screens: extrude on the side stream, under SH_step's
    // remaining kernels (which are still running or queued on `st`), and join before the optics
    AOG_CUDA(cudaStreamWaitEvent(env->side_stream, env->ev_sh_phase, 0));
    rc = evolve_to(env, env->cnt.timestep, old_t, noise_dev, env->side_stream);
    if (rc) return rc;
    AOG_CUDA(cudaEventRecord(env->ev_ext_done, env->side_stream));
    AOG_CUDA(cudaStreamWaitEvent(st, env->ev_ext_done, 0));
  } else {
    rc = evolve_to(env, env->cnt.timestep, old_t, noise_dev, st);
    if (rc) return rc;
  }
  env->sh_phase_pending = false;
  if (env->timing) {
    AOG_CUDA(cudaEventRecord(env->tev[1], st));
    env->last_extrusions = (int)(env->cnt.extrusions - ext_before);
    env->tev_ext_valid = true;
  }
  // AO_env.py:132-144
  aog_outputs o{};
  if (out_dev) o = *out_dev;
  rc = optics_all(env, false, true, o, st);
  if (rc) return rc;
  // AO_env.py:147-151
  int done = 0;
  if (env->cnt.timestep_render == c.max_steps) { done = 1; env->cnt.episode_no += 1; }
  if (done_out) *done_out = done;
  return AOG_OK;
}

int aog_step_host(aog_env* env, const void* actions_host, int act_dtype, const double* noise_host,
                  const aog_outputs* out_host, int32_t* done_out) {
  if (!env || !actions_host) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  AOG_DEVICE(c.device);
  cudaStream_t st = env->own_stream;
  if (act_dtype != AOG_DTYPE_F32 && act_dtype != AOG_DTYPE_F64) AOG_FAIL(AOG_ERR_INVALID, "act_dtype");
  const size_t esz = act_dtype == AOG_DTYPE_F32 ? sizeof(float) : sizeof(double);
  const size_t abytes = (size_t)c.num_envs * c.num_modes * esz;
  // Small batches on a static atmosphere: the whole step (H2D, kernels, D2H) is a CUDA graph captured on the second
  // call and relaunched afterwards -- the step of a single env is launch-bound (4 kernels + 2 copies).
  const bool no_graph = getenv("AOG_NO_GRAPH") != nullptr;
  if (c.num_envs <= 256 && c.precision != AOG_PRECISION_F64 && c.velocity == 0.0 && !noise_host && !env->timing &&
      !env->graph_failed && !no_graph && tables_ready(env)) {
    int rc;
    if (!env->h_act) AOG_CUDA(cudaMallocHost(&env->h_act, (size_t)c.num_envs * c.num_modes * sizeof(double)));
    if ((rc = ensure_pinned(env, env->o_pack_bytes))) return rc;
    std::memcpy(env->h_act, actions_host, abytes);
    aog_outputs d = device_outputs(env);
    if (env->step_graph && env->graph_dtype == act_dtype) {
      // host bookkeeping of aog_step (AO_env.py:123-124, 147-151); the device work is the graph
      env->cnt.timestep += 1;
      env->cnt.timestep_render += 1;
      int done = 0;
      if (env->cnt.timestep_render == c.max_steps) { done = 1; env->cnt.episode_no += 1; }
      if (done_out) *done_out = done;
      AOG_CUDA(cudaGraphLaunch(env->step_graph, st));
      env->launches += env->graph_launches;
    } else if (env->graph_warm >= 1) {
      if (env->step_graph) { cudaGraphExecDestroy(env->step_graph); env->step_graph = nullptr; }
      cudaGraph_t graph = nullptr;
      const int64_t l0 = env->launches;
      AOG_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      cudaError_t e = cudaMemcpyAsync(env->act_in, env->h_act, abytes, cudaMemcpyHostToDevice, st);
      rc = e == cudaSuccess ? aog_step(env, env->act_in, act_dtype, nullptr, &d, done_out, st) : AOG_ERR_CUDA;
      if (rc == AOG_OK) e = cudaMemcpyAsync(env->h_pinned, env->o_pack, env->o_pack_bytes, cudaMemcpyDeviceToHost, st);
      const cudaError_t e2 = cudaStreamEndCapture(st, &graph);
      if (rc != AOG_OK || e != cudaSuccess || e2 != cudaSuccess || !graph ||
          cudaGraphInstantiate(&env->step_graph, graph, 0) != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        env->step_graph = nullptr;
        env->graph_failed = true;                      // this handle keeps to plain launches
        if (rc != AOG_OK) return rc;                   // (aog_step's own error; its bookkeeping has not been undone)
        AOG_FAIL(AOG_ERR_CUDA, "CUDA graph capture of the step failed");
      }
      cudaGraphDestroy(graph);
      env->graph_dtype = act_dtype;
      env->graph_launches = (int)(env->launches - l0);
      AOG_CUDA(cudaGraphLaunch(env->step_graph, st));  // the capture recorded the work, this runs it
    } else {
      env->graph_warm++;                               // first call: plain launches (function attributes, lazy set-up)
      AOG_CUDA(cudaMemcpyAsync(env->act_in, env->h_act, abytes, cudaMemcpyHostToDevice, st));
      if ((rc = aog_step(env, env->act_in, act_dtype, nullptr, &d, done_out, st))) return rc;
      AOG_CUDA(cudaMemcpyAsync(env->h_pinned, env->o_pack, env->o_pack_bytes, cudaMemcpyDeviceToHost, st));
    }
    AOG_CUDA(cudaStreamSynchronize(st));
    scatter_host_outputs(env, out_host);
    return AOG_OK;
  }
  AOG_CUDA(cudaMemcpyAsync(env->act_in, actions_host, abytes, cudaMemcpyHostToDevice, st));
  const double* nz = nullptr;
  if (noise_host) {
    const int n_ext = aog_next_extrusions(env);
    const size_t cnt = (size_t)c.num_envs * n_ext * c.num_pupil_pixels;
    if (cnt > 0) {
      if (cnt > env->noise_in_cap) {
        int rc = dev_alloc(env, &env->noise_in, cnt);
        if (rc) return rc;
        env->noise_in_cap = cnt;
      }
      AOG_CUDA(cudaMemcpyAsync(env->noise_in, noise_host, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
      nz = env->noise_in;
    }
  }
  aog_outputs d = device_outputs(env);
  int rc = aog_step(env, env->act_in, act_dtype, nz, &d, done_out, st);
  if (rc) return rc;
  return copy_outputs_to_host(env, out_host, st);
}

int aog_sh_configure(aog_env* env, int num_sub, int num_pix, double amplitude, double weight_dt) {
  if (!env) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (num_sub < 1 || num_pix < num_sub || num_pix > env->P) AOG_FAIL(AOG_ERR_INVALID, "Shack-Hartmann sizes");
  AOG_DEVICE(c.device);
  const size_t P = env->P, K = c.num_modes, B = c.num_envs;
  env->sh_num_sub = num_sub;
  env->sh_num_pix = num_pix;
  env->sh_amplitude = amplitude;
  env->sh_weight_dt = weight_dt;
  int rc;
#define A(expr) if ((rc = (expr))) return rc
  A(dev_alloc(env, &env->t_sh_mla, P));
  A(dev_alloc(env, &env->t_sh_C, P));
  A(dev_alloc(env, &env->t_sh_CT, P));
  A(dev_alloc(env, &env->t_sh_off, (size_t)num_sub + 1));
  A(dev_alloc(env, &env->t_sh_pix, (size_t)num_pix));
  A(dev_alloc(env, &env->t_sh_px, (size_t)num_pix));
  A(dev_alloc(env, &env->t_sh_py, (size_t)num_pix));
  A(dev_alloc(env, &env->t_sh_offset, 2 * (size_t)num_sub));
  A(dev_alloc(env, &env->t_sh_recon, K * 2 * (size_t)num_sub));
  A(dev_alloc(env, &env->t_sh_act0, K));
  A(dev_alloc(env, &env->act_sh, B * K));
  A(dev_alloc(env, &env->o_action, B * K));
#undef A
  AOG_CUDA(cudaMemset(env->act_sh, 0, B * K * sizeof(double)));
  for (int t = AOG_TABLE_SH_MLA_PHASE; t <= AOG_TABLE_SH_ACT0; ++t) env->have[t] = false;
  return AOG_OK;
}

// AO_env.py:254-290 for every env of the handle: atmosphere + the SH mirror + micro-lens array (k_sh_field_f64),
// Fresnel propagation to the lenslet focal plane as E_out = C E C^T (two batched complex GEMMs), then camera
// image, photon noise, centroids, slopes and the leaky-integrator update (k_sh_centroid_update).
int aog_sh_step(aog_env* env, int noise_mode, const double* noisy_image_dev, double* action_out_dev, void* stream) {
  if (!env) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (env->sh_num_sub == 0) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
  for (int t = AOG_TABLE_SH_MLA_PHASE; t <= AOG_TABLE_SH_ACT0; ++t)
    if (!env->have[t]) AOG_FAIL(AOG_ERR_STATE, "Shack-Hartmann table " + std::to_string(t) + " not set");
  if (!env->have[AOG_TABLE_APERTURE] || !env->have[AOG_TABLE_DM_MODES]) AOG_FAIL(AOG_ERR_STATE, "tables not set");
  if (noise_mode < AOG_SH_NOISE_NONE || noise_mode > AOG_SH_NOISE_INJECTED) AOG_FAIL(AOG_ERR_INVALID, "noise_mode");
  if (noise_mode == AOG_SH_NOISE_INJECTED && !noisy_image_dev) AOG_FAIL(AOG_ERR_INVALID, "noisy image missing");
  AOG_DEVICE(c.device);
  cudaStream_t st = (cudaStream_t)stream;
  if (c.precision != AOG_PRECISION_F64 && noise_mode != AOG_SH_NOISE_INJECTED) {
    // tensor / fused precision: the Fresnel products on tcgen05, FP32 camera (sh_tensor.cuh); tables without the
    // structure those kernels need fall through to the FP64 kernels below
    const int trc = aog_tensor_sh_step(env, noise_mode, action_out_dev, st);
    if (trc == AOG_OK) { env->sh_draws++; return AOG_OK; }
    if (trc != AOG_ERR_UNSUPPORTED) return trc;
  }
  int rc = ensure_f64_scratch(env);
  if (rc) return rc;
  const int Np = c.num_pupil_pixels, K = c.num_modes, P = env->P, B = c.num_envs, Nsub = env->sh_num_sub;
  const long long sB = (long long)Np * std::max(c.num_focal_pixels, Np);
  const long long sC = (long long)std::max<size_t>(env->NF2, P);
  constexpr int ET = 4;
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    const double2* F = env->bufC;
    long long strideF = sC;
    if (noise_mode != AOG_SH_NOISE_INJECTED && env->sh_fold) {
      // parity-folded Fresnel step: four (Np/2)^3 products per stage instead of one Np^3 (common.cuh: t_sh_Cf)
      const int Nh = Np / 2, Q = Nh * Nh;
      const long long blk = (long long)env->chunk * Q;
      constexpr int EF = 4;                  // envs per thread (8 measured slower: 6.2 vs ~4 ms, register pressure)
      k_sh_field_fold<EF><<<dim3(cdiv(Q, 128), cdiv(nB, EF)), 128, EF * K * sizeof(double), st>>>(
          env->screens, env->act_sh, env->t_modes, env->t_aperture, env->t_sh_mla, env->bufA, blk, P, Np, K, e0, nB,
          (int)env->cnt.column_origin, c.wavelength_wfs, env->sh_amplitude);
      AOG_LAUNCH_CHECK();
      const dim3 g(cdiv(Nh, 64), cdiv(Nh, 64), nB);
      for (int b = 0; b < 4; ++b) {          // Y_pq = C_p E_pq
        k_zgemm<<<g, 256, 0, st>>>(env->t_sh_Cf[b >> 1], env->bufA + b * blk, env->bufB + b * blk, Nh, Nh, Nh, Nh, Nh, Nh,
                                   0, (long long)Q, (long long)Q);
        AOG_LAUNCH_CHECK();
      }
      for (int b = 0; b < 4; ++b) {          // G_pq = Y_pq C_q^T
        k_zgemm<<<g, 256, 0, st>>>(env->bufB + b * blk, env->t_sh_Cf[2 + (b & 1)], env->bufC + b * blk, Nh, Nh, Nh, Nh, Nh,
                                   Nh, (long long)Q, 0, (long long)Q);
        AOG_LAUNCH_CHECK();
      }
      k_sh_unfold<<<dim3(cdiv(Q, 128), nB), 128, 0, st>>>(env->bufC, blk, env->bufA, Np, nB);
      AOG_LAUNCH_CHECK();
      F = env->bufA;
      strideF = P;
    } else if (noise_mode != AOG_SH_NOISE_INJECTED) {
      k_sh_field_f64<ET><<<dim3(cdiv(P, 128), cdiv(nB, ET)), 128, ET * K * sizeof(double), st>>>(
          env->screens, env->act_sh, env->t_modes, env->t_aperture, env->t_sh_mla, env->bufA, P, Np, K, e0, nB,
          (int)env->cnt.column_origin, c.wavelength_wfs, env->sh_amplitude);
      AOG_LAUNCH_CHECK();
      k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->t_sh_C, env->bufA, env->bufB, Np, Np, Np, Np,
                                                                     Np, Np, 0, (long long)P, sB);
      AOG_LAUNCH_CHECK();
      k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), nB), 256, 0, st>>>(env->bufB, env->t_sh_CT, env->bufC, Np, Np, Np, Np,
                                                                     Np, Np, sB, 0, sC);
      AOG_LAUNCH_CHECK();
    }
    k_sh_centroid_update<<<nB, 256, 2 * Nsub * sizeof(double), st>>>(
        F, strideF, env->t_sh_off, env->t_sh_pix, env->t_sh_px, env->t_sh_py, env->t_sh_offset, env->t_sh_recon,
        env->act_sh, action_out_dev, noisy_image_dev, P, K, Nsub, e0, env->sh_weight_dt, noise_mode,
        c.seed ^ 0xD1B54A32D192ED03ull, (unsigned long long)c.env_id_base, (unsigned long long)env->sh_draws);
    AOG_LAUNCH_CHECK();
  }
  env->sh_draws++;
  return AOG_OK;
}

int aog_sh_step_host(aog_env* env, int noise_mode, const double* noisy_image_host, double* action_out_host) {
  if (!env || !action_out_host) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  AOG_DEVICE(c.device);
  cudaStream_t st = env->own_stream;
  const size_t B = c.num_envs, K = c.num_modes, P = env->P;
  if (!env->o_action) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
  const double* noisy = nullptr;
  if (noise_mode == AOG_SH_NOISE_INJECTED) {
    if (!noisy_image_host) AOG_FAIL(AOG_ERR_INVALID, "noisy image missing");
    if (!env->sh_noisy_in) { int rc = dev_alloc(env, &env->sh_noisy_in, B * P); if (rc) return rc; }
    AOG_CUDA(cudaMemcpyAsync(env->sh_noisy_in, noisy_image_host, B * P * sizeof(double), cudaMemcpyHostToDevice, st));
    noisy = env->sh_noisy_in;
  }
  int rc = aog_sh_step(env, noise_mode, noisy, env->o_action, st);
  if (rc) return rc;
  AOG_CUDA(cudaMemcpyAsync(action_out_host, env->o_action, B * K * sizeof(double), cudaMemcpyDeviceToHost, st));
  AOG_CUDA(cudaStreamSynchronize(st));
  return AOG_OK;
}

int aog_get_counters(const aog_env* env, aog_counters* out) {
  if (!env || !out) return AOG_ERR_INVALID;
  *out = env->cnt;
  out->screen_draws = env->screen_draws;
  out->sh_draws = env->sh_draws;
  return AOG_OK;
}

int aog_set_counters(aog_env* env, const aog_counters* in) {
  if (!env || !in) return AOG_ERR_INVALID;
  env->cnt = *in;
  env->screen_draws = in->screen_draws;
  env->sh_draws = in->sh_draws;
  return AOG_OK;
}

int aog_reseed(aog_env* env, uint64_t seed) {
  if (!env) return AOG_ERR_INVALID;
  env->cfg.seed = seed;
  env->cnt.extrusions = 0;      // the three Philox offset domains restart under the new key
  env->screen_draws = 0;
  env->sh_draws = 0;
  return AOG_OK;
}

int aog_health(aog_env* env) {
  if (!env) return AOG_ERR_INVALID;
  return aog_tensor_check(env);
}

int aog_get_sh_actuators(aog_env* env, double* host_out) {
  if (!env || !host_out) return AOG_ERR_INVALID;
  if (!env->act_sh) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
  AOG_DEVICE(env->cfg.device);
  AOG_CUDA(cudaDeviceSynchronize());
  AOG_CUDA(cudaMemcpy(host_out, env->act_sh, (size_t)env->cfg.num_envs * env->cfg.num_modes * sizeof(double),
                      cudaMemcpyDeviceToHost));
  return AOG_OK;
}

int aog_set_sh_actuators(aog_env* env, const double* host_in) {
  if (!env || !host_in) return AOG_ERR_INVALID;
  if (!env->act_sh) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
  AOG_DEVICE(env->cfg.device);
  AOG_CUDA(cudaDeviceSynchronize());
  AOG_CUDA(cudaMemcpy(env->act_sh, host_in, (size_t)env->cfg.num_envs * env->cfg.num_modes * sizeof(double),
                      cudaMemcpyHostToDevice));
  return AOG_OK;
}

int aog_get_actuators(aog_env* env, double* host_out) {
  if (!env || !host_out) return AOG_ERR_INVALID;
  AOG_DEVICE(env->cfg.device);
  AOG_CUDA(cudaDeviceSynchronize());
  AOG_CUDA(cudaMemcpy(host_out, env->act, (size_t)env->cfg.num_envs * env->cfg.num_modes * sizeof(double),
                      cudaMemcpyDeviceToHost));
  return AOG_OK;
}

int aog_set_actuators(aog_env* env, const double* host_in) {
  if (!env || !host_in) return AOG_ERR_INVALID;
  AOG_DEVICE(env->cfg.device);
  AOG_CUDA(cudaDeviceSynchronize());
  AOG_CUDA(cudaMemcpy(env->act, host_in, (size_t)env->cfg.num_envs * env->cfg.num_modes * sizeof(double),
                      cudaMemcpyHostToDevice));
  return AOG_OK;
}

int aog_get_field(aog_env* env, int which, int env_index, double* host_out, size_t count) {
  if (!env || !host_out) return AOG_ERR_INVALID;
  const aog_config& c = env->cfg;
  if (env_index < 0 || env_index >= c.num_envs) AOG_FAIL(AOG_ERR_INVALID, "env_index");
  if (!tables_ready(env)) return AOG_ERR_STATE;
  AOG_DEVICE(c.device);
  AOG_CUDA(cudaDeviceSynchronize());
  const size_t P = env->P;
  if (which == AOG_FIELD_SCREEN) {
    if (count != P) AOG_FAIL(AOG_ERR_INVALID, "count");
    return aog_get_screens(env, host_out, env_index, 1);
  }
  if (which == AOG_FIELD_ACTUATORS) {
    if (count != (size_t)c.num_modes) AOG_FAIL(AOG_ERR_INVALID, "count");
    AOG_CUDA(cudaMemcpy(host_out, env->act + (size_t)env_index * c.num_modes, count * sizeof(double),
                        cudaMemcpyDeviceToHost));
    return AOG_OK;
  }
  if (which == AOG_FIELD_SH_ACTUATORS) {
    if (!env->act_sh) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
    if (count != (size_t)c.num_modes) AOG_FAIL(AOG_ERR_INVALID, "count");
    AOG_CUDA(cudaMemcpy(host_out, env->act_sh + (size_t)env_index * c.num_modes, count * sizeof(double),
                        cudaMemcpyDeviceToHost));
    return AOG_OK;
  }
  if (which == AOG_FIELD_SH_IMAGE_TC) {   // the same image through the tensor-core kernels (tests)
    if (c.precision == AOG_PRECISION_F64) AOG_FAIL(AOG_ERR_INVALID, "tensor-path field on an FP64 handle");
    if (!env->act_sh) AOG_FAIL(AOG_ERR_STATE, "aog_sh_configure not called");
    return aog_tensor_sh_image(env, env_index, host_out, count);
  }
  if (which == AOG_FIELD_SH_IMAGE) {   // noise-free camera image (power x dt) for the current state
    if (!env->act_sh || !env->have[AOG_TABLE_SH_FRESNEL] || !env->have[AOG_TABLE_SH_MLA_PHASE])
      AOG_FAIL(AOG_ERR_STATE, "Shack-Hartmann tables not set");
    if (count != P) AOG_FAIL(AOG_ERR_INVALID, "count");
    int rc = ensure_f64_scratch(env);
    if (rc) return rc;
    const int Np = c.num_pupil_pixels, K = c.num_modes;
    cudaStream_t st = env->own_stream;
    k_sh_field_f64<1><<<dim3(cdiv((int)P, 128), 1), 128, K * sizeof(double), st>>>(
        env->screens, env->act_sh, env->t_modes, env->t_aperture, env->t_sh_mla, env->bufA, (int)P, Np, K, env_index,
        1, (int)env->cnt.column_origin, c.wavelength_wfs, env->sh_amplitude);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), 1), 256, 0, st>>>(env->t_sh_C, env->bufA, env->bufB, Np, Np, Np, Np, Np,
                                                                  Np, 0, 0, 0);
    AOG_LAUNCH_CHECK();
    k_zgemm<<<dim3(cdiv(Np, 64), cdiv(Np, 64), 1), 256, 0, st>>>(env->bufB, env->t_sh_CT, env->bufC, Np, Np, Np, Np, Np,
                                                                  Np, 0, 0, 0);
    AOG_LAUNCH_CHECK();
    std::vector<double> f(2 * P);
    AOG_CUDA(cudaMemcpyAsync(f.data(), env->bufC, 2 * P * sizeof(double), cudaMemcpyDeviceToHost, st));
    AOG_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < P; ++i) host_out[i] = (f[2 * i] * f[2 * i] + f[2 * i + 1] * f[2 * i + 1]) * env->sh_weight_dt;
    return AOG_OK;
  }
  if (which == AOG_FIELD_TC_PUPIL || which == AOG_FIELD_TC_STAGE1) {
    if (c.precision != AOG_PRECISION_TENSOR) AOG_FAIL(AOG_ERR_INVALID, "tensor-path field: the handle has no matrix-Fourier-transform GEMM stages");
    return aog_tensor_get_field(env, which, env_index % env->chunk, host_out, count);
  }
  // optical fields: recompute the FP64 chain for that one env from the current state
  { int rc = ensure_f64_scratch(env); if (rc) return rc; }
  aog_outputs d = device_outputs(env);
  aog_outputs none{};
  none.obs_f64 = d.obs_f64;   // optics_chunk_f64 applies the env offset itself
  const bool timing = env->timing;
  env->timing = false;
  int rc = optics_chunk_f64(env, env_index, 1, false, false, none, env->own_stream);
  env->timing = timing;
  if (rc) return rc;
  AOG_CUDA(cudaStreamSynchronize(env->own_stream));
  if (which == AOG_FIELD_PUPIL) {
    if (count != 2 * P) AOG_FAIL(AOG_ERR_INVALID, "count");
    AOG_CUDA(cudaMemcpy(host_out, env->bufA, count * sizeof(double), cudaMemcpyDeviceToHost));
  } else if (which == AOG_FIELD_FOCAL || which == AOG_FIELD_FOCAL_POWER) {
    const size_t nf2 = env->NF2;
    std::vector<double> f(2 * nf2);
    AOG_CUDA(cudaMemcpy(f.data(), env->bufC, 2 * nf2 * sizeof(double), cudaMemcpyDeviceToHost));
    const double nr = c.mft_norm_re, ni = c.mft_norm_im;
    const double w = (c.obs_weight * c.obs_dim * c.obs_dim) / (double)nf2;   // same window, Nf^2 pixels
    if (which == AOG_FIELD_FOCAL) {
      if (count != 2 * nf2) AOG_FAIL(AOG_ERR_INVALID, "count");
      for (size_t i = 0; i < nf2; ++i) {
        host_out[2 * i] = f[2 * i] * nr - f[2 * i + 1] * ni;
        host_out[2 * i + 1] = f[2 * i] * ni + f[2 * i + 1] * nr;
      }
    } else {
      if (count != nf2) AOG_FAIL(AOG_ERR_INVALID, "count");
      for (size_t i = 0; i < nf2; ++i) {
        const double fr = f[2 * i] * nr - f[2 * i + 1] * ni, fi = f[2 * i] * ni + f[2 * i + 1] * nr;
        host_out[i] = (fr * fr + fi * fi) * w;
      }
    }
  } else if (which == AOG_FIELD_OBS_POWER) {
    if (count != (size_t)env->n2) AOG_FAIL(AOG_ERR_INVALID, "count");
    AOG_CUDA(cudaMemcpy(host_out, d.obs_f64 + (size_t)env_index * env->n2, count * sizeof(double), cudaMemcpyDeviceToHost));
  } else {
    AOG_FAIL(AOG_ERR_INVALID, "unknown field");
  }
  return AOG_OK;
}

int aog_debug_poisson(int device, double lambda, int n, uint64_t seed, double* host_out) {
  if (!host_out || n < 1 || !(lambda >= 0.0)) return AOG_ERR_INVALID;
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return AOG_ERR_CUDA;
  double* d = nullptr;
  if (cudaMalloc((void**)&d, (size_t)n * sizeof(double)) != cudaSuccess) return AOG_ERR_CUDA;
  k_debug_poisson<<<cdiv(n, 256), 256>>>(lambda, n, (unsigned long long)seed, d);
  const cudaError_t e = cudaMemcpy(host_out, d, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(d);
  return e == cudaSuccess ? AOG_OK : AOG_ERR_CUDA;
}

int aog_debug_poisson_f32(int device, double lambda, int n, uint64_t seed, double* host_out) {
  if (!host_out || n < 1 || !(lambda >= 0.0)) return AOG_ERR_INVALID;
  return aog_tensor_debug_poisson(device, lambda, n, seed, host_out);
}

int aog_debug_normals(int device, int generator, int philox, int n, const uint32_t* words_in, uint32_t* raw_out,
                      float* normals_out) {
  if (!words_in || !normals_out || (philox && !raw_out) || n < 1 || (generator != 0 && generator != 1))
    return AOG_ERR_INVALID;
  return aog_tensor_debug_normals(device, generator, philox, n, words_in, raw_out, normals_out);
}

int64_t aog_launch_count(const aog_env* env) { return env ? env->launches : -1; }

int aog_chunk_size(const aog_env* env) { return env ? env->chunk : AOG_ERR_INVALID; }

int aog_set_timing(aog_env* env, int enabled) {
  if (!env) return AOG_ERR_INVALID;
  env->timing = enabled != 0;
  env->ev_valid = false;
  env->tev_ext_valid = env->tev_sh_valid = false;
  return AOG_OK;
}

int aog_last_kernel_ms(aog_env* env, double* field_ms, double* stage1_ms, double* stage2_ms) {
  if (!env) return AOG_ERR_INVALID;
  if (!env->ev_valid || env->cfg.precision == AOG_PRECISION_F64) AOG_FAIL(AOG_ERR_STATE, "no timed tensor-path step yet");
  AOG_CUDA(cudaEventSynchronize(env->ev1));
  float a = 0.f, b = 0.f, c = 0.f;
  AOG_CUDA(cudaEventElapsedTime(&a, env->evf, env->ev0));
  AOG_CUDA(cudaEventElapsedTime(&b, env->ev0, env->evm));
  AOG_CUDA(cudaEventElapsedTime(&c, env->evm, env->ev1));
  if (field_ms) *field_ms = a;
  if (stage1_ms) *stage1_ms = b;
  if (stage2_ms) *stage2_ms = c;
  return AOG_OK;
}

int aog_last_timings(aog_env* env, double* out_ms, int n) {
  if (!env || !out_ms || n < 7) return AOG_ERR_INVALID;
  for (int i = 0; i < n; ++i) out_ms[i] = -1.0;
  float ms = 0.f;
  if (env->tev_ext_valid) {
    AOG_CUDA(cudaEventSynchronize(env->tev[1]));
    AOG_CUDA(cudaEventElapsedTime(&ms, env->tev[0], env->tev[1]));
    out_ms[0] = ms;
    out_ms[1] = (double)env->last_extrusions;
  }
  if (env->tev_sh_valid) {
    AOG_CUDA(cudaEventSynchronize(env->tev[7]));
    for (int k = 0; k < 5; ++k) {
      AOG_CUDA(cudaEventElapsedTime(&ms, env->tev[2 + k], env->tev[3 + k]));
      out_ms[2 + k] = ms;
    }
  }
  return AOG_OK;
}

double aog_last_mft_ms(aog_env* env) {
  if (!env || !env->ev_valid) return -1.0;
  if (cudaEventSynchronize(env->ev1) != cudaSuccess) return -1.0;
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, env->ev0, env->ev1) != cudaSuccess) return -1.0;
  return (double)ms;
}

}  // extern "C"
