// The arguments of the per-env epilogue, shared by k_finalize (FP64 path, kernels_f64.cuh) and k_finalize_tcw
// (tensor / fused paths, tensor_path.cu), and ssim_1d, the SSIM k_finalize computes and k_finalize_tcw reproduces.
#pragma once
#include "common.cuh"

struct FinalizeArgs {
  const double2* R; const float2* R4; const double2* m1o; const double2* coef; const double* coef4; const double2* lpphase; const double* lpgram;
  const double2* strehl_part; int strehl_blocks;
  int Np, n, J, rew_type, has_thr, compute_reward;
  int coef_is_raw;     // 2: coef4 holds [re|im][2 partials]; 3: fib_part holds [fib_slots][fib_stride] partial sums
                       // per env;  both x coef_scale
  const double2* fib_part; int fib_slots, fib_stride;
  // the phase kernel's CTA c takes work items [c slot_ipc, (c + 1) slot_ipc) and the 128-env block eb owns items
  // [eb slot_items, (eb + 1) slot_items), so only slots 0 .. last - first of an env are written (and summed): no
  // clearing pass
  int slot_ipc, slot_items;
  // the env's normalised actuators [K].  An all-zero action makes them 0/0 = NaN (AO_env.py:119-120) and the
  // reference then returns NaN observations, reward and power; the fixed-point phase arithmetic of the tensor / fused
  // kernels would swallow the NaN, so it is re-applied here.
  const double* act; int K;
  double2 coef_scale;
  double thr, obs_weight, strehl_scale, ssim_peak;
  double2 norm;
  uint16_t* obs16; double* obs64; double* reward; double* power; double* strehl; double* ssim;
};

__device__ __forceinline__ double ssim_1d(const double* x, int len, int ref_idx, double peak) {
  // skimage.metrics.structural_similarity 0.22 on 1-D data against peak * onehot(ref_idx):
  // win 7, uniform filter, sample covariance, K1 = .01, K2 = .03, crop 3, mean.
  const double C1 = (0.01 * peak) * (0.01 * peak), C2 = (0.03 * peak) * (0.03 * peak);
  const double cov_norm = 7.0 / 6.0;
  double tot = 0.0;
  for (int c = 3; c < len - 3; ++c) {
    double sx = 0, sxx = 0, sy = 0, syy = 0, sxy = 0;
    for (int i = c - 3; i <= c + 3; ++i) {
      const double a = x[i], r = (i == ref_idx) ? peak : 0.0;
      sx += a; sxx += a * a; sy += r; syy += r * r; sxy += a * r;
    }
    const double ux = sx / 7, uy = sy / 7, uxx = sxx / 7, uyy = syy / 7, uxy = sxy / 7;
    const double vx = cov_norm * (uxx - ux * ux), vy = cov_norm * (uyy - uy * uy), vxy = cov_norm * (uxy - ux * uy);
    tot += ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
  }
  return tot / (double)(len - 6);
}
