// FP64 (exact) kernels of the AO-v0 step path.  This is the guaranteed-parity arithmetic
// (AOG_PRECISION_F64) and the on-device checker for the tensor-core path.
#pragma once
#include "fft240.cuh"
#include "common.cuh"
#include "finalize.cuh"
#include "philox.cuh"
#include <curand_kernel.h>

// --------------------------------------------------------------------------------------
// Action normalisation (reference AO_env.py:115-120):
//   a = action / (arange(K) + 10);  a *= 0.1 lambda_sci / std(M a),  std^2 = a^T G a
// One block per env.
// --------------------------------------------------------------------------------------
template <typename ActT>
static __global__ void k_actuators(const ActT* __restrict__ actions, const double* __restrict__ gram,
                            double* __restrict__ act, int K, int sh_operation, double target_rms) {
  extern __shared__ double sh_a[];   // [K] + [32] reduction scratch
  double* red = sh_a + K;
  const int b = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    double a = (double)actions[(size_t)b * K + k];
    sh_a[k] = sh_operation ? a : a / (double)(k + 10);
  }
  __syncthreads();
  if (sh_operation) {
    for (int k = threadIdx.x; k < K; k += blockDim.x) act[(size_t)b * K + k] = sh_a[k];
    return;
  }
  double part = 0.0;
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    double r = 0.0;
    for (int j = 0; j < K; ++j) r += gram[(size_t)j * K + i] * sh_a[j];   // G is symmetric: read it column-wise (coalesced)
    part += sh_a[i] * r;
  }
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x < 32) {
    double v = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.0;
    v = warp_sum(v);
    if (threadIdx.x == 0) red[0] = v;
  }
  __syncthreads();
  // var == 0 -> inf -> 0 * inf = NaN (reference semantics).  The Gram matrix is singular (duplicated disk-harmonic
  // modes): for an action in its null space rounding can leave var slightly negative, where np.std is >= 0
  const double scale = target_rms / sqrt(fmax(red[0], 0.0));
  for (int k = threadIdx.x; k < K; k += blockDim.x) act[(size_t)b * K + k] = sh_a[k] * scale;
}

// --------------------------------------------------------------------------------------
// DM surface + pupil field + Strehl partial sums (AO_env.py:132-135, 479-483):
//   s = M a;  E = amp A exp(i (S / l_wfs + 2 s k_wfs));  sum_ap exp(i (S / l_sci + 2 s k_sci))
// Thread = one pixel for ET envs (the mode value is loaded once and reused ET times).
// grid (ceil(P/128), ceil(nB/ET)), block 128.
// --------------------------------------------------------------------------------------
template <int ET>
static __global__ void k_field_f64(const double* __restrict__ screens, const double* __restrict__ act,
                            const double* __restrict__ modes, const double* __restrict__ aperture,
                            double2* __restrict__ E, double2* __restrict__ strehl_part, int P, int Np, int K,
                            int env0, int nB, int col_origin, double l_wfs, double l_sci, double amp,
                            int do_strehl, int flat_dm) {
  extern __shared__ double sh_act[];   // [ET][K]
  __shared__ double2 red[ET][4];
  const int e0 = blockIdx.y * ET;
  for (int i = threadIdx.x; i < ET * K; i += blockDim.x) {
    int e = i / K, k = i - e * K;
    sh_act[i] = (e0 + e < nB && !flat_dm) ? act[(size_t)(env0 + e0 + e) * K + k] : 0.0;
  }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = p < P;
  double s[ET];
#pragma unroll
  for (int e = 0; e < ET; ++e) s[e] = 0.0;
  if (valid && !flat_dm) {
    for (int k = 0; k < K; ++k) {
      const double m = modes[(size_t)k * P + p];
#pragma unroll
      for (int e = 0; e < ET; ++e) s[e] = fma(m, sh_act[e * K + k], s[e]);
    }
  }
  const double ap = valid ? aperture[p] : 0.0;
  int y = 0, xp = 0;
  if (valid) {
    y = p / Np;
    xp = p - y * Np + col_origin;
    if (xp >= Np) xp -= Np;
  }
  const double kw = 6.283185307179586476925286766559 / l_wfs;
  const double ks = 6.283185307179586476925286766559 / l_sci;
#pragma unroll
  for (int e = 0; e < ET; ++e) {
    double2 st = make_double2(0.0, 0.0);
    if (valid && e0 + e < nB) {
      const double S = screens[(size_t)(env0 + e0 + e) * P + (size_t)xp * Np + y];
      double sn, cs;
      sincos(S / l_wfs + 2.0 * s[e] * kw, &sn, &cs);
      E[(size_t)(e0 + e) * P + p] = make_double2(amp * ap * cs, amp * ap * sn);
      if (do_strehl) {
        sincos(S / l_sci + 2.0 * s[e] * ks, &sn, &cs);
        st = make_double2(ap * cs, ap * sn);
      }
    }
    if (do_strehl) {
      st.x = warp_sum(st.x);
      st.y = warp_sum(st.y);
      if ((threadIdx.x & 31) == 0) red[e][threadIdx.x >> 5] = st;
    }
  }
  if (do_strehl) {
    __syncthreads();
    if (threadIdx.x < ET && e0 + threadIdx.x < nB) {
      double2 a = red[threadIdx.x][0];
      for (int w = 1; w < 4; ++w) { a.x += red[threadIdx.x][w].x; a.y += red[threadIdx.x][w].y; }
      strehl_part[(size_t)(e0 + threadIdx.x) * gridDim.x + blockIdx.x] = a;
    }
  }
}

// --------------------------------------------------------------------------------------
// Batched complex FP64 GEMM  C[b] = A[b] (M x Kd) . B[b] (Kd x N), row-major, stride 0 = shared.
// 64x64x16 tiles, 256 threads, 4x4 complex accumulators per thread.
// --------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) k_zgemm(const double2* __restrict__ A, const double2* __restrict__ B,
                                               double2* __restrict__ C, int M, int N, int Kd, int lda, int ldb,
                                               int ldc, long long sA, long long sB, long long sC) {
  __shared__ double2 As[16][65];
  __shared__ double2 Bs[16][64];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  A += (size_t)blockIdx.z * sA;
  B += (size_t)blockIdx.z * sB;
  C += (size_t)blockIdx.z * sC;
  double2 acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_double2(0.0, 0.0);
  const double2 zero = make_double2(0.0, 0.0);
  for (int k0 = 0; k0 < Kd; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = threadIdx.x & 15, m = (threadIdx.x >> 4) + 16 * i;
      As[k][m] = (m0 + m < M && k0 + k < Kd) ? A[(size_t)(m0 + m) * lda + k0 + k] : zero;
      const int n = threadIdx.x & 63, kb = (threadIdx.x >> 6) + 4 * i;
      Bs[kb][n] = (n0 + n < N && k0 + kb < Kd) ? B[(size_t)(k0 + kb) * ldb + n0 + n] : zero;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      double2 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j].x = fma(a[i].x, b[j].x, acc[i][j].x);
          acc[i][j].x = fma(-a[i].y, b[j].y, acc[i][j].x);
          acc[i][j].y = fma(a[i].x, b[j].y, acc[i][j].y);
          acc[i][j].y = fma(a[i].y, b[j].x, acc[i][j].y);
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty + 16 * i, n = n0 + tx + 16 * j;
      if (m < M && n < N) C[(size_t)m * ldc + n] = acc[i][j];
    }
}

// --------------------------------------------------------------------------------------
// Fibre-mode projection (AO_env.py:471): c_j = norm * sum_q F[q] (mode_j w)[q].  Block per env.
// --------------------------------------------------------------------------------------
static __global__ void k_fiber_f64(const double2* __restrict__ F, const double* __restrict__ lpw,
                            double2* __restrict__ coef, int NF2, int J, long long strideF, double2 norm) {
  __shared__ double2 red[AOG_MAX_LP][8];
  const int b = blockIdx.x;
  const double2* f = F + (size_t)b * strideF;
  double2 acc[AOG_MAX_LP];
#pragma unroll
  for (int j = 0; j < AOG_MAX_LP; ++j) acc[j] = make_double2(0.0, 0.0);
  for (int q = threadIdx.x; q < NF2; q += blockDim.x) {
    const double2 v = f[q];
#pragma unroll
    for (int j = 0; j < AOG_MAX_LP; ++j)
      if (j < J) {
        const double w = lpw[(size_t)j * NF2 + q];
        acc[j].x = fma(v.x, w, acc[j].x);
        acc[j].y = fma(v.y, w, acc[j].y);
      }
  }
#pragma unroll
  for (int j = 0; j < AOG_MAX_LP; ++j)
    if (j < J) {
      acc[j].x = warp_sum(acc[j].x);
      acc[j].y = warp_sum(acc[j].y);
      if ((threadIdx.x & 31) == 0) red[j][threadIdx.x >> 5] = acc[j];
    }
  __syncthreads();
  if (threadIdx.x < J) {
    double2 a = make_double2(0.0, 0.0);
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a.x += red[threadIdx.x][w].x; a.y += red[threadIdx.x][w].y; }
    coef[(size_t)b * J + threadIdx.x] = make_double2(a.x * norm.x - a.y * norm.y, a.x * norm.y + a.y * norm.x);
  }
}

// --------------------------------------------------------------------------------------
// Photodetector arm, first contraction (AO_env.py:139): R[y][u] = sum_x E[y][x] M2o[x][u].
// Warp per pupil row; grid (ceil(Np/8), nB), block 256.
// --------------------------------------------------------------------------------------
static __global__ void k_obs_rows_f64(const double2* __restrict__ E, const double2* __restrict__ m2o,
                               double2* __restrict__ R, int Np, int n, int P) {
  const int y = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (y >= Np) return;
  const double2* row = E + (size_t)blockIdx.y * P + (size_t)y * Np;
  for (int u = 0; u < n; ++u) {
    double re = 0.0, im = 0.0;
    for (int x = lane; x < Np; x += 32) {
      const double2 e = row[x], m = m2o[(size_t)x * n + u];
      re += e.x * m.x - e.y * m.y;
      im += e.x * m.y + e.y * m.x;
    }
    re = warp_sum(re);
    im = warp_sum(im);
    if (lane == 0) R[((size_t)blockIdx.y * Np + y) * n + u] = make_double2(re, im);
  }
}

// --------------------------------------------------------------------------------------
// Per-env epilogue: obs power (second contraction + |.|^2 w), fibre power, Strehl, SSIM,
// reward, threshold (AO_env.py:142-153, 468-503).  k_finalize (FP64 path, block per env) reads R and coef;
// k_finalize_tcw (tensor / fused paths, warp per env, tensor_path.cu) reads R4 and the partial sums and actuators
// described in finalize.cuh.
// --------------------------------------------------------------------------------------
static __global__ void k_finalize(FinalizeArgs a) {
  __shared__ double obs[AOG_MAX_OBS * AOG_MAX_OBS];
  const int b = blockIdx.x;
  const int n2 = a.n * a.n;
  // one warp per photodetector pixel, lanes split the contraction index, FP64 accumulation
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int t = warp; t < n2; t += nwarps) {
    const int v = t / a.n, u = t - v * a.n;
    double re = 0.0, im = 0.0;
    const double2* r = a.R + (size_t)b * a.Np * a.n;
    for (int y = lane; y < a.Np; y += 32) {
      const double2 m = a.m1o[(size_t)v * a.Np + y], e = r[(size_t)y * a.n + u];
      re += m.x * e.x - m.y * e.y;
      im += m.x * e.y + m.y * e.x;
    }
    re = warp_sum(re);
    im = warp_sum(im);
    if (lane == 0) {
      const double fr = re * a.norm.x - im * a.norm.y, fi = re * a.norm.y + im * a.norm.x;
      const double pw = (fr * fr + fi * fi) * a.obs_weight;
      obs[t] = pw;
      if (a.obs64) a.obs64[(size_t)b * n2 + t] = pw;
      if (a.obs16) a.obs16[(size_t)b * n2 + t] = __half_as_ushort(__double2half(pw));
    }
  }
  __syncthreads();
  if (threadIdx.x != 0 || !a.compute_reward) return;
  // fibre: out = M (c e^{i beta L});  total power = c'^H G c'
  double2 c[AOG_MAX_LP];
  for (int j = 0; j < a.J; ++j) {
    const double2 cj = a.coef[(size_t)b * a.J + j];
    const double2 ph = a.lpphase[j];
    c[j] = make_double2(cj.x * ph.x - cj.y * ph.y, cj.x * ph.y + cj.y * ph.x);
  }
  double power = 0.0;
  for (int j = 0; j < a.J; ++j)
    for (int k = 0; k < a.J; ++k)
      power += a.lpgram[j * a.J + k] * (c[j].x * c[k].x + c[j].y * c[k].y);
  double reward;
  if (a.rew_type == AOG_REW_STREHL_RATIO) {
    double sr = 0.0, si = 0.0;
    const double2* sp = a.strehl_part + (size_t)b * a.strehl_blocks;
#pragma unroll 8
    for (int i = 0; i < a.strehl_blocks; ++i) { sr += sp[i].x; si += sp[i].y; }
    const double strehl = a.strehl_scale * (sr * sr + si * si);
    if (a.strehl) a.strehl[b] = strehl;
    reward = -(100.0 - strehl);
  } else {
    const double s = ssim_1d(obs, n2, n2 / 2, a.ssim_peak);
    if (a.ssim) a.ssim[b] = s;
    reward = 0.8 * power + (1.0 - 0.8) * s;
  }
  if (a.has_thr && reward < a.thr) reward = -1.0;
  if (a.reward) a.reward[b] = reward;
  if (a.power) a.power[b] = power;
}

// --------------------------------------------------------------------------------------
// Autoregressive column extrusion (hcipy InfiniteAtmosphericLayer._extrude; AO_env.py:125).
// gather: Z[b] = [ screen[stencil] (on the 180-degree rotated screen when moving +x) ,
//                  sqrt(Cn2) xi ];  GEMM: new = Z . [A^T ; B^T];  scatter: ring slot.
// --------------------------------------------------------------------------------------
// extrusion noise: normals 4 j .. 4 j + 3 of extrusion `draw` of env `env_id`
__device__ __forceinline__ void ar_normals4(unsigned long long seed, unsigned long long env_id, unsigned long long draw,
                                            int j, float (&z)[4]) {
  aog_normals4(aog_philox4x32_10(make_uint4((uint32_t)j, (uint32_t)draw, (uint32_t)(draw >> 32), (uint32_t)env_id),
                                 make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(env_id >> 32))), z);
}

static __global__ void k_ar_gather(const double* __restrict__ screens, const int* __restrict__ stencil,
                            const double* __restrict__ noise, double* __restrict__ Z, int P, int Np, int Ns,
                            int env0, int col_origin, int flipped, const double* __restrict__ sqrt_cn2,
                            long long noise_stride, unsigned long long seed, unsigned long long env_id_base,
                            unsigned long long draw_index) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Ns + Np) return;
  double v;
  if (j < Ns) {
    int q = stencil[j];
    int y = q / Np, x = q - y * Np;
    if (flipped) { y = Np - 1 - y; x = Np - 1 - x; }
    x += col_origin;
    if (x >= Np) x -= Np;
    v = screens[(size_t)(env0 + b) * P + (size_t)x * Np + y];
  } else {
    const int i = j - Ns;
    double xi;
    if (noise) {
      xi = noise[(size_t)(env0 + b) * noise_stride + i];
    } else {
      // one Philox block makes four normals: threads i, i ^ 1, i ^ 2, i ^ 3 share the block i / 4 (as k_ar_noise draws them)
      float z[4];
      ar_normals4(seed, env_id_base + env0 + b, draw_index, i >> 2, z);
      xi = (double)z[i & 3];
    }
    v = sqrt_cn2[env0 + b] * xi;
  }
  Z[(size_t)b * (Ns + Np) + j] = v;
}

// sqrt(Cn2) xi for ALL the extrusions of a step in one launch (the DIRECT form of k_ar_step reads it in place):
// NZ[(e nB + b) Np + i], e < next;  the same Philox draws as k_ar_gather (extrusion e uses draw index draw0 + e), one
// block per four normals, or the injected normals noise[(env0 + b) noise_stride + e Np + i].
static __global__ void k_ar_noise(const double* __restrict__ noise, double* __restrict__ NZ, int Np, int nB, int next,
                                  int env0, const double* __restrict__ sqrt_cn2, long long noise_stride, unsigned long long seed,
                                  unsigned long long env_id_base, unsigned long long draw0) {
  const int b = blockIdx.y, e = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = 4 * j;
  if (i >= Np) return;
  const double s = sqrt_cn2[env0 + b];         // loaded first: its latency hides under the Philox rounds
  double v[4];
  if (noise) {
    const double* src = noise + (size_t)(env0 + b) * noise_stride + (size_t)e * Np + i;
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = i + k < Np ? src[k] : 0.0;
  } else {
    float z[4];
    ar_normals4(seed, env_id_base + env0 + b, draw0 + e, j, z);
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (double)z[k];
  }
  double* dst = NZ + ((size_t)e * nB + b) * Np + i;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (i + k < Np) dst[k] = s * v[k];
}

// new column = Z . W (hcipy _extrude: A z + B xi for every env) on the FP64 tensor cores, with the scatter into the
// ring-buffered screens -- and, for the tensor / fused paths, the refresh of that column's fixed-point phase tiles --
// in the epilogue.  mma.sync.m8n8k4.f64 (DMMA) sustains 36 TFLOP/s on B200 with 4-8 warps per SM where scalar DFMA
// needs 16+ warps of 32 independent chains for 31 (tools/micro/dmma_bench.cu), and it issues 8x fewer instructions,
// which leaves the slots for the operand traffic.  Block tile 128 envs x 64 pixels, warp tile 32 x 32 = 4 x 4
// fragments.  ncu: DMMA pipe 50 % of the active cycles, 128 blocks on 148 SMs; splitting K over a second group of
// 8 warps per tile (dmma_mainloop<2>) measured no gain (140 vs 135 us), so the plain form is used.
//   screens[(env0 + b) P + phys_col Np + y] = new[b][flipped ? Np - 1 - y : y]      (screens are [x][y]: a column is contiguous)
//   tiles (TensorState::hwt layout) [env / 32][phys_col][y / 16][env % 32][piece][y % 4] = fixed(new / (lambda_wfs pi))
// Main loop shared by the FP64 tensor-core GEMMs: acc (warp tile 32 x 32 at (wm, wn) of the 128 x 64 block tile at
// (m0, n0)) = A[M x Kd] (row stride lda) . B[Kd x N] (row stride ldb).  lda, ldb, Kd, N even, rows 16-byte aligned.
// Operands stream global -> shared with 16-byte cp.async through a DMMA_STAGES-deep ring of K steps of 8 * KSPLIT (no
// register staging, no transposing stores): A keeps its row-major form, rows padded by 4 doubles so that a fragment
// load (8 rows x 4 consecutive k) touches every bank once; B rows padded to 68.
// KSPLIT = 2 (512 threads): two groups of 8 warps work on the SAME output tile, group g on the k range
// [8 g, 8 g + 8) of every K step, and the second group's accumulators are added through shared memory at the end --
// 16 warps per SM for a GEMM whose grid has fewer blocks than the GPU has SMs (the extrusion: 128 blocks).
constexpr int DMMA_STAGES = 4, DMMA_LDB = 64 + 4;
template <int KSPLIT> struct DmmaCfg {
  static constexpr int TK = 8 * KSPLIT, LDA = TK + 4, A_STAGE = 128 * LDA, B_STAGE = TK * DMMA_LDB;   // doubles
  static constexpr int RING = DMMA_STAGES * (A_STAGE + B_STAGE) * (int)sizeof(double);
  static constexpr int SMEM = KSPLIT == 2 ? (RING > 65536 ? RING : 65536) : RING;       // ring, reused for the reduction
  static constexpr int THREADS = 256 * KSPLIT;
};
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool ok) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int n = ok ? 16 : 0;                                   // src-size 0: the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
// returns true for the threads that hold the finished tile (group 0)
template <int KSPLIT>
__device__ __forceinline__ bool dmma_mainloop(const double* __restrict__ A, int lda, int M, const double* __restrict__ B,
                                              int ldb, int N, int Kd, int m0, int n0, double (&acc)[4][4][2]) {
  using Cfg = DmmaCfg<KSPLIT>;
  constexpr int TK = Cfg::TK, LDA = Cfg::LDA;
  extern __shared__ __align__(16) double dmma_smem[];
  double* As = dmma_smem;                                      // [stage][128][LDA]
  double* Bs = dmma_smem + DMMA_STAGES * Cfg::A_STAGE;         // [stage][TK][DMMA_LDB]
  const int group = threadIdx.x >> 8, t = threadIdx.x & 255;
  const int warp = t >> 5, lane = t & 31, gid = lane >> 2, tig = lane & 3;
  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;      // warp tile origin inside the block tile
  // loader roles (group g loads the k range it will use): A row t / 2, k pairs 2 (t % 2) + {0, 1};  B row t / 32, n pair t % 32
  const int am = t >> 1, ac = (t & 1) * 2, kg = group * 8;
  const int bk = t >> 5, bc = t & 31;
  const bool a_ok = m0 + am < M, b_ok = n0 + 2 * bc < N;
  const double* a_src = A + (size_t)(a_ok ? m0 + am : 0) * lda;
  const double* b_src = B + (b_ok ? n0 + 2 * bc : 0);
  auto issue = [&](int ks) {                                   // K step ks -> ring slot ks % DMMA_STAGES
    const int k0 = ks * TK + kg, st = ks % DMMA_STAGES;
    double* as = As + st * Cfg::A_STAGE + am * LDA + kg;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int k = k0 + 2 * (ac + c);
      cp_async16(as + 2 * (ac + c), a_src + (k < Kd ? k : 0), a_ok && k < Kd);
    }
    const int kb = k0 + bk;
    cp_async16(Bs + st * Cfg::B_STAGE + (kg + bk) * DMMA_LDB + 2 * bc, b_src + (size_t)(kb < Kd ? kb : 0) * ldb, b_ok && kb < Kd);
  };
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int nk = (Kd + TK - 1) / TK;
#pragma unroll
  for (int s0 = 0; s0 < DMMA_STAGES - 1; ++s0) {
    if (s0 < nk) issue(s0);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int ks = 0; ks < nk; ++ks) {
    asm volatile("cp.async.wait_group %0;" ::"n"(DMMA_STAGES - 2) : "memory");   // K step ks has landed
    __syncthreads();                                            // ... for every thread; slot (ks - 1) % STAGES is free
    if (ks + DMMA_STAGES - 1 < nk) issue(ks + DMMA_STAGES - 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const double* as = As + (ks % DMMA_STAGES) * Cfg::A_STAGE + kg;
    const double* bs = Bs + (ks % DMMA_STAGES) * Cfg::B_STAGE + kg * DMMA_LDB;
#pragma unroll
    for (int k4 = 0; k4 < 8; k4 += 4) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = as[(wm + 8 * i + gid) * LDA + k4 + tig];          // A fragment: row gid, column (k) tig
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = bs[(k4 + tig) * DMMA_LDB + wn + 8 * j + gid];     // B fragment: row (k) tig, column gid
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                       : "+d"(acc[i][j][0]), "+d"(acc[i][j][1]) : "d"(a[i]), "d"(b[j]));
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (KSPLIT == 2) {
    __syncthreads();                                            // the ring is dead: reuse it for the second group's tile
    double* red = dmma_smem + (size_t)t * 32;
    if (group == 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<double2*>(red + (i * 4 + j) * 2) = make_double2(acc[i][j][0], acc[i][j][1]);
    }
    __syncthreads();
    if (group == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double2 v = *reinterpret_cast<const double2*>(red + (i * 4 + j) * 2);
          acc[i][j][0] += v.x;
          acc[i][j][1] += v.y;
        }
    }
  }
  return group == 0;
}

// Batched real FP64 GEMM on the tensor cores: C_z[M x N] = A_z[M x Kd] . B_z[Kd x N], z = blockIdx.z, operand z at
// base + z * stride (stride 0 = shared table).  Grid (ceil(N / 64), ceil(M / 128), batch).
static __global__ void __launch_bounds__(256)
k_dgemm_mma(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ C, int M, int N, int Kd,
            int lda, int ldb, int ldc, long long sA, long long sB, long long sC) {
  const int m0 = blockIdx.y * 128, n0 = blockIdx.x * 64;
  double acc[4][4][2];
  dmma_mainloop<1>(A + (size_t)blockIdx.z * sA, lda, M, B + (size_t)blockIdx.z * sB, ldb, N, Kd, m0, n0, acc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
  double* c = C + (size_t)blockIdx.z * sC;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + wm + 8 * i + gid;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + wn + 8 * j + 2 * tig;
      if (n + 1 < N) *reinterpret_cast<double2*>(&c[(size_t)m * ldc + n]) = make_double2(acc[i][j][0], acc[i][j][1]);
      else if (n < N) c[(size_t)m * ldc + n] = acc[i][j][0];
    }
  }
}

// The extrusion GEMM's own tiling: 112 envs x 64 pixels per block, 7 warps of 16 x 64 (2 x 8 fragments).  4096 envs
// are 37 x 4 = 148 such tiles -- one per SM of a B200 in a single wave (the shared 128 x 64 tile gave 128 blocks).
constexpr int AR_TM = 112, AR_THREADS = 224, AR_LDA = 8 + 4, AR_A_STAGE = AR_TM * AR_LDA, AR_B_STAGE = 8 * DMMA_LDB;
constexpr int AR_SMEM = DMMA_STAGES * (AR_A_STAGE + AR_B_STAGE) * (int)sizeof(double);
// DIRECT (round 2): the A operand is read where it lives instead of from a gathered copy Z (k_ar_gather: 24 us per
// extrusion, launch-shape bound).  In gather order the stencil is [column 0 | column 1 | one pixel per row further
// back | noise]: the two newest columns are contiguous runs of the column-major screens (16-byte cp.async, in MEMORY
// order -- for the rotated screen of a +x extrusion that is the reversed row order, so W has a second copy with
// those rows reversed), the Np tail pixels are single doubles (8-byte cp.async at the geometric offsets), and the
// scaled normals of ALL extrusions of a step come from one k_ar_noise launch.  The column this launch overwrites is
// the oldest one (logical column Np - 1), which the upload code checks is not in the stencil.
struct ArDirect {
  const double* nz;      // [nB][Np] sqrt(Cn2) xi of this extrusion (chunk-relative rows)
  const int* tail;       // [Ns - 2 Np] (x | y << 16) logical coordinates of the tail pixels, gather order
  int pc0, pc1;          // physical columns of stencil columns 0 and 1
  int org, Ns;
};
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc, bool ok) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int n = ok ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
template <bool DIRECT>
static __global__ void __launch_bounds__(AR_THREADS)
k_ar_step(const double* __restrict__ Z, const double* __restrict__ W, double* __restrict__ screens,
          int32_t* __restrict__ tiles, int nB, int Np, int Kd, int P, int env0, int phys_col, int flipped,
          double inv_w, double phi_one, ArDirect dr) {
  extern __shared__ __align__(16) double dmma_smem[];
  double* As = dmma_smem;                                      // [stage][112][AR_LDA]
  double* Bs = dmma_smem + DMMA_STAGES * AR_A_STAGE;           // [stage][8][DMMA_LDB]
  const int m0 = blockIdx.y * AR_TM, n0 = blockIdx.x * 64;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, gid = lane >> 2, tig = lane & 3;
  const int wm = warp * 16;
  // DIRECT loader: this thread's two A rows (t / 4 and t / 4 + 56) and its k pair inside a K step
  const int lrow = t >> 2, lkc = (t & 3) * 2;
  const bool ok0 = m0 + lrow < nB, ok1 = m0 + lrow + AR_THREADS / 4 < nB;
  const double* scr0 = screens + (size_t)(env0 + (ok0 ? m0 + lrow : 0)) * P;
  const double* scr1 = screens + (size_t)(env0 + (ok1 ? m0 + lrow + AR_THREADS / 4 : 0)) * P;
  const double* nz0 = DIRECT ? dr.nz + (size_t)(ok0 ? m0 + lrow : 0) * Np : nullptr;
  const double* nz1 = DIRECT ? dr.nz + (size_t)(ok1 ? m0 + lrow + AR_THREADS / 4 : 0) * Np : nullptr;
  int* tail_off = reinterpret_cast<int*>(dmma_smem + DMMA_STAGES * (AR_A_STAGE + AR_B_STAGE));   // [Ns - 2 Np] offsets into an env's screen
  if constexpr (DIRECT) {
    for (int j = t; j < dr.Ns - 2 * Np; j += AR_THREADS) {
      const int xy = __ldg(dr.tail + j);
      int x = xy & 0xffff, y = xy >> 16;
      if (flipped) { x = Np - 1 - x; y = Np - 1 - y; }
      x += dr.org;
      if (x >= Np) x -= Np;
      tail_off[j] = x * Np + y;
    }
    __syncthreads();
  }
  auto issue = [&](int ks) {                                   // K step ks (8 deep) -> ring slot ks % DMMA_STAGES
    const int k0 = ks * 8, st = ks % DMMA_STAGES;
    if constexpr (DIRECT) {
      const int k = k0 + lkc;
      double* d0 = As + st * AR_A_STAGE + lrow * AR_LDA + lkc;
      double* d1 = d0 + (AR_THREADS / 4) * AR_LDA;
      const bool kok = k < Kd;
      if (k < 2 * Np) {                                        // the two newest columns, memory order
        const int off = k < Np ? dr.pc0 * Np + k : dr.pc1 * Np + (k - Np);
        cp_async16(d0, scr0 + off, ok0);
        cp_async16(d1, scr1 + off, ok1);
      } else if (k < dr.Ns) {                                  // tail pixels: one double each
        const int2 off = *reinterpret_cast<const int2*>(tail_off + (k - 2 * Np));
        cp_async8(d0, scr0 + off.x, ok0);
        cp_async8(d0 + 1, scr0 + off.y, ok0);
        cp_async8(d1, scr1 + off.x, ok1);
        cp_async8(d1 + 1, scr1 + off.y, ok1);
      } else {                                                 // noise
        const int off = kok ? k - dr.Ns : 0;
        cp_async16(d0, nz0 + off, ok0 && kok);
        cp_async16(d1, nz1 + off, ok1 && kok);
      }
    } else {
#pragma unroll
    for (int i = 0; i < 2; ++i) {                              // A: 112 rows x 4 chunks of 2 doubles
      const int c = t + AR_THREADS * i, row = c >> 2, kc = (c & 3) * 2;
      const bool ok = m0 + row < nB && k0 + kc < Kd;
      cp_async16(As + st * AR_A_STAGE + row * AR_LDA + kc, Z + (size_t)(ok ? m0 + row : 0) * Kd + (ok ? k0 + kc : 0), ok);
    }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {                              // B: 8 rows x 32 chunks of 2 doubles
      const int c = t + AR_THREADS * i;
      if (c < 256) {
        const int row = c >> 5, nc = (c & 31) * 2;
        const bool ok = k0 + row < Kd && n0 + nc < Np;
        cp_async16(Bs + st * AR_B_STAGE + row * DMMA_LDB + nc, W + (size_t)(ok ? k0 + row : 0) * Np + (ok ? n0 + nc : 0), ok);
      }
    }
  };
  double acc[2][8][2];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int nk = (Kd + 7) / 8;
#pragma unroll
  for (int s0 = 0; s0 < DMMA_STAGES - 1; ++s0) {
    if (s0 < nk) issue(s0);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int ks = 0; ks < nk; ++ks) {
    asm volatile("cp.async.wait_group %0;" ::"n"(DMMA_STAGES - 2) : "memory");   // K step ks has landed
    __syncthreads();                                            // ... for every thread; slot (ks - 1) % STAGES is free
    if (ks + DMMA_STAGES - 1 < nk) issue(ks + DMMA_STAGES - 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const double* as = As + (ks % DMMA_STAGES) * AR_A_STAGE;
    const double* bs = Bs + (ks % DMMA_STAGES) * AR_B_STAGE;
#pragma unroll
    for (int k4 = 0; k4 < 8; k4 += 4) {
      double a[2], b[8];
#pragma unroll
      for (int i = 0; i < 2; ++i) a[i] = as[(wm + 8 * i + gid) * AR_LDA + k4 + tig];
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = bs[(k4 + tig) * DMMA_LDB + 8 * j + gid];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                       : "+d"(acc[i][j][0]), "+d"(acc[i][j][1]) : "d"(a[i]), "d"(b[j]));
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  // C fragment: row gid, columns 2 tig + {0, 1}
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int b = m0 + wm + 8 * i + gid;
    if (b >= nB) continue;
    const size_t env = (size_t)env0 + b;
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int e2 = 0; e2 < 2; ++e2) {
        const int n = n0 + 8 * j + 2 * tig + e2;
        if (n >= Np) continue;
        const int y = flipped ? Np - 1 - n : n;
        const double S = acc[i][j][e2];
        screens[env * P + (size_t)phys_col * Np + y] = S;          // the ring slot is one contiguous column
        if (tiles) {
          double f = S * inv_w * phi_one;
          f = fmin(fmax(f, -2147483000.0), 2147483000.0);
          const int l = (int)(env & 31), ci = y >> 4, piece = ((y >> 2) & 3) ^ ((l >> 1) & 3), e = y & 3;
          const size_t tile = (((env >> 5) * Np + phys_col) * (size_t)(Np / 16) + ci) * 512;
          tiles[tile + (size_t)l * 16 + piece * 4 + e] = (int32_t)__double2ll_rn(f);
        }
      }
  }
}

// --------------------------------------------------------------------------------------
// von-Karman screen synthesis (semi_dynamic reset; AO_env.py:76-77): spectral noise
// X = C . (xi_r + i xi_i), then screen = Re[W X W^T] through the batched complex GEMM.
// --------------------------------------------------------------------------------------
// Spectral normals of the synthesis: ONE Philox-4x32-10 block (counter = element pair, env; key = seed) makes the two
// complex normals of elements 2 j and 2 j + 1 by two Box-Muller transforms in FP32 on the SFU (24-bit uniforms,
// lg2 / sqrt / sin / cos approximations: a normal deviate good to ~1e-6, |z| <= 5.9) -- the screens are random draws,
// equivalent to the reference's only statistically, and curand's FP64 Box-Muller (log, sqrt, sincospi in double, one
// curand_init per element) was 2.6 ms of a 10.7 ms reset of 4096 envs.
// z[0..3]: (re, im) of element 2 j, (re, im) of element 2 j + 1;  pair = (draw_base + i) / 2 for even i
__device__ __forceinline__ void scr_normals4(unsigned long long seed, unsigned long long env_id, unsigned long long pair,
                                             float (&z)[4]) {
  aog_normals4(aog_philox4x32_10(make_uint4((uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)env_id, (uint32_t)(env_id >> 32)),
                                 make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))), z);
}
static __global__ void k_scr_noise(const double* __restrict__ C, double2* __restrict__ X, int count, long long strideX,
                            int env0, unsigned long long seed, unsigned long long env_id_base,
                            unsigned long long draw_base) {
  const int b = blockIdx.y;
  const int i = 2 * (blockIdx.x * blockDim.x + threadIdx.x);                // count and draw_base are even
  if (i >= count) return;
  float z[4];
  scr_normals4(seed, env_id_base + env0 + b, (draw_base + (unsigned long long)i) >> 1, z);
  const double c0 = C[i], c1 = C[i + 1];
  X[(size_t)b * strideX + i] = make_double2(c0 * (double)z[0], c0 * (double)z[1]);
  X[(size_t)b * strideX + i + 1] = make_double2(c1 * (double)z[2], c1 * (double)z[3]);
}

// FFT form of the fine scale (fft240.cuh): S1 = Re IDFT2(X sh sh^T) for Np = 240, W1[x][k] = sh[k] w^(x k).
//   k_scr_fft_rows: T[ky][x] = sum_kx X'[ky][kx] w^(x kx),  X' = (Xr + i Xi) sh[ky] sh[kx]     (FFT_LINES rows per block)
//   k_scr_fft_cols: screens[x][y] (+)= scale Re sum_ky T[ky][x] w^(y ky)                        (FFT_LINES columns per block)
// X is generated inside the row kernel (the Philox draws of k_scr_noise_planes, so the GEMM forms give the same
// screens); the column kernel writes the screens, and the coarse scale's k_scr_combine4 then adds its part and writes
// the fixed-point phase tiles of the tensor / fused paths (the column kernel can do both itself -- `accumulate`,
// `tiles` -- but its few warps hide the read-modify-write badly: 2.6 ms against 1.9 + 0.4 in the element-wise kernel).  256 threads: stage 1 on 16 x 15 threads, stage 2 on 16 x 16; the 240-slot line buffers
// sit in shared memory (rows padded for the column kernel's transposing stores).
#ifndef AOG_FFT_LINES
#define AOG_FFT_LINES 16
#endif
constexpr int FFT_LINES = AOG_FFT_LINES, FFT_THREADS = 16 * FFT_LINES, FFT_LD = 241;
constexpr int FFT_SMEM = (FFT_LINES * FFT_LD + 2 * 240) * (int)sizeof(double2);
static __global__ void __launch_bounds__(FFT_THREADS)
k_scr_fft_rows(const double* __restrict__ C, const double2* __restrict__ sh, const double2* __restrict__ tw,
               double2* __restrict__ T, long long sT, int env0, unsigned long long seed, unsigned long long env_id_base,
               unsigned long long draw_base) {
  constexpr int N = 240;
  extern __shared__ __align__(16) double2 fft_smem[];
  double2* buf = fft_smem;                       // [16][FFT_LD]
  double2* tw_s = fft_smem + FFT_LINES * FFT_LD; // [240]
  double2* sh_s = tw_s + N;                      // [240]
  const int b = blockIdx.y, ky0 = blockIdx.x * FFT_LINES, t = threadIdx.x;
  for (int i = t; i < N; i += FFT_THREADS) { tw_s[i] = tw[i]; sh_s[i] = sh[i]; }
  __syncthreads();
  // X = C . xi: the draws of k_scr_noise_planes (element i = ky N + kx, pairs of elements per Philox block), never stored
  for (int pi = t; pi < FFT_LINES * (N / 2); pi += FFT_THREADS) {
    const int r = pi / (N / 2), kx = 2 * (pi - r * (N / 2)), ky = ky0 + r, i = ky * N + kx;
    float z[4];
    scr_normals4(seed, env_id_base + env0 + b, (draw_base + (unsigned long long)i) >> 1, z);
    const double c0 = C[i], c1 = C[i + 1];
    const double2 s0 = fft240::cmul(sh_s[ky], sh_s[kx]), s1 = fft240::cmul(sh_s[ky], sh_s[kx + 1]);
    buf[r * FFT_LD + kx] = fft240::cmul(make_double2(c0 * (double)z[0], c0 * (double)z[1]), s0);
    buf[r * FFT_LD + kx + 1] = fft240::cmul(make_double2(c1 * (double)z[2], c1 * (double)z[3]), s1);
  }
  __syncthreads();
  if (t < FFT_LINES * 15) fft240::stage1(buf + (t / 15) * FFT_LD, 1, t % 15, tw_s);
  __syncthreads();
  {
    // T is stored [ky / 16][x][ky % 16]: this block's 16 rows are the 16 contiguous entries of every x, so the column
    // kernel reads 4 KB runs (a plain [ky][x] layout made it gather 256-byte pieces at a 3840-byte stride: 3.2 ms)
    static_assert(FFT_LINES == 16, "T layout");
    const int r = t & 15, k1 = t >> 4;
    double2 a[15];
    fft240::stage2(buf + r * FFT_LD, 1, k1, a);
    double2* out = T + (size_t)b * sT + ((size_t)blockIdx.x * N + k1) * 16 + r;
#pragma unroll
    for (int k2 = 0; k2 < 15; ++k2) out[(size_t)16 * k2 * 16] = a[k2];
  }
}
static __global__ void __launch_bounds__(FFT_THREADS)
k_scr_fft_cols(const double2* __restrict__ T, long long sT, const double2* __restrict__ tw, double* __restrict__ screens,
               int P, int env0, const double* __restrict__ sqrt_cn2, int accumulate, int32_t* __restrict__ tiles,
               double inv_w, double phi_one) {
  constexpr int N = 240;
  extern __shared__ __align__(16) double2 fft_smem[];
  double2* buf = fft_smem;                       // [16 columns][FFT_LD]
  double2* tw_s = fft_smem + FFT_LINES * FFT_LD;
  const int b = blockIdx.y, x0 = blockIdx.x * FFT_LINES, t = threadIdx.x;
  const double scale = sqrt_cn2[env0 + b];
  for (int i = t; i < N; i += FFT_THREADS) tw_s[i] = tw[i];
  const double2* tb = T + (size_t)b * sT;
  {
    double2 v[N / 16];                                 // all 15 loads in flight before the first store
#pragma unroll
    for (int kb = 0; kb < N / 16; ++kb) v[kb] = tb[((size_t)kb * N + x0) * 16 + t];   // T is [ky / 16][x][ky % 16]: 16 columns x 16 rows = one 4 KB run
#pragma unroll
    for (int kb = 0; kb < N / 16; ++kb) buf[(t >> 4) * FFT_LD + kb * 16 + (t & 15)] = v[kb];
  }
  __syncthreads();
  if (t < FFT_LINES * 15) fft240::stage1(buf + (t / 15) * FFT_LD, 1, t % 15, tw_s);
  __syncthreads();
  {
    const int c = t >> 4, k1 = t & 15;
    double2 a[15];
    fft240::stage2(buf + c * FFT_LD, 1, k1, a);
    double* out = screens + (size_t)(env0 + b) * P + (size_t)(x0 + c) * N + k1;     // screens are [x][y]
    // the finished screen's fixed-point phase tile (TensorState::hwt, as k_ar_step's epilogue writes it): y = k1 + 16 k2
    // is element k1 of chunk k2, column origin 0 after a synthesis
    const size_t env = (size_t)env0 + b;
    const int l = (int)(env & 31), piece = ((k1 >> 2) & 3) ^ ((l >> 1) & 3), e = k1 & 3;
    int32_t* trow = tiles ? tiles + (((env >> 5) * N + (x0 + c)) * (size_t)(N / 16)) * 512 + (size_t)l * 16 + piece * 4 + e : nullptr;
#pragma unroll
    for (int k2 = 0; k2 < 15; ++k2) {
      double v = scale * a[k2].x;
      if (accumulate) v += out[16 * k2];
      out[16 * k2] = v;
      if (tiles) {
        double f = v * inv_w * phi_one;
        f = fmin(fmax(f, -2147483000.0), 2147483000.0);
        trow[(size_t)k2 * 512] = (int32_t)__double2ll_rn(f);
      }
    }
  }
}

// real-arithmetic synthesis (common.cuh: t_scrWst): the same draws as k_scr_noise, written as two real planes
// X[b] = [Xr | Xi], Nk rows of 2 Nk doubles
static __global__ void k_scr_noise_planes(const double* __restrict__ C, double* __restrict__ X, int Nk, long long strideX,
                                          int env0, unsigned long long seed, unsigned long long env_id_base,
                                          unsigned long long draw_base) {
  const int b = blockIdx.y;
  const int i = 2 * (blockIdx.x * blockDim.x + threadIdx.x);                // Nk and draw_base are even
  if (i >= Nk * Nk) return;
  float z[4];
  scr_normals4(seed, env_id_base + env0 + b, (draw_base + (unsigned long long)i) >> 1, z);
  const double c0 = C[i], c1 = C[i + 1];
  const int k = i / Nk, l = i - k * Nk;                                     // i + 1 is in the same row
  double* x = X + (size_t)b * strideX + (size_t)k * 2 * Nk + l;
  x[0] = c0 * (double)z[0];
  x[Nk] = c0 * (double)z[1];
  x[1] = c1 * (double)z[2];
  x[Nk + 1] = c1 * (double)z[3];
}

// S at the four mirror images of (y, x), y, x < N/2, from P1 = Ur Wr^T, P2 = Vi Wr^T, P3 = Ui Wi^T, P4 = Vr Wi^T
// (U = Re W_top X, V = Im W_top X): (P1 -+ P2) -+ (P3 +- P4)
// tiles != null (the last writer of a synthesis): also the fixed-point phase tiles of the tensor / fused paths
// (TensorState::hwt, as k_ar_step's epilogue writes them; column origin 0)
static __global__ void k_scr_combine4(double* __restrict__ screens, const double* __restrict__ Pq, int Np,
                                      long long strideP, int env0, const double* __restrict__ sqrt_cn2, int accumulate,
                                      int32_t* __restrict__ tiles, double inv_w, double phi_one) {
  const int Nh = Np / 2, Q = Nh * Nh;
  const int b = blockIdx.y;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const int x = q / Nh, y = q - x * Nh;                // consecutive threads -> consecutive y: contiguous stores
  const double* p = Pq + (size_t)b * strideP + (size_t)y * Nh + x;
  const double p1 = p[0], p2 = p[Q], p3 = p[2 * Q], p4 = p[3 * Q];
  double* s = screens + (size_t)(env0 + b) * Np * Np;  // [x][y]
  const double v[4] = {(p1 - p2) - (p3 + p4), (p1 - p2) + (p3 + p4), (p1 + p2) - (p3 - p4), (p1 + p2) + (p3 - p4)};
  const size_t idx[4] = {(size_t)x * Np + y, (size_t)(Np - 1 - x) * Np + y, (size_t)x * Np + (Np - 1 - y),
                         (size_t)(Np - 1 - x) * Np + (Np - 1 - y)};
  const size_t env = (size_t)env0 + b;
  const double scale = sqrt_cn2[env];
  const int l = (int)(env & 31);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const double out = accumulate ? (s[idx[c]] + scale * v[c]) : scale * v[c];
    s[idx[c]] = out;
    if (tiles) {
      const int xx = (int)(idx[c] / Np), yy = (int)(idx[c] - (size_t)xx * Np);
      double f = out * inv_w * phi_one;
      f = fmin(fmax(f, -2147483000.0), 2147483000.0);
      tiles[(((env >> 5) * Np + xx) * (size_t)(Np / 16) + (yy >> 4)) * 512 + (size_t)l * 16 +
            ((((yy >> 2) & 3) ^ ((l >> 1) & 3)) << 2) + (yy & 3)] = (int32_t)__double2ll_rn(f);
    }
  }
}

// aog_set_turbulence's rescale on an FP64 handle: screens[b][*] *= factor[b] (the tensor / fused handles do this in
// k_screens_to_tiles, which also rewrites the phase tiles)
static __global__ void k_scale_screens(double* __restrict__ screens, const double* __restrict__ factor, int P,
                                       size_t total) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) screens[i] *= factor[i / P];
}

static __global__ void k_scr_combine(double* __restrict__ screens, const double2* __restrict__ Y, int P, long long strideY,
                              int env0, const double* __restrict__ sqrt_cn2, int accumulate) {
  const int b = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  // thread p = (x, y) with y fastest (contiguous stores into the column-major screens); Y is [y][x]
  int Np = 1;
  while (Np * Np < P) ++Np;
  const int x = p / Np, y = p - x * Np;
  const double v = sqrt_cn2[env0 + b] * Y[(size_t)b * strideY + (size_t)y * Np + x].x;
  double* s = screens + (size_t)(env0 + b) * P + p;
  *s = accumulate ? (*s + v) : v;
}

// --------------------------------------------------------------------------------------
// Shack-Hartmann integrator (AO_env.py:254-290).
// field: E = amp A exp(i (S / l_wfs + 2 k s_sh + mla_phase)),  s_sh = M a_sh  (atmosphere, the SH mirror,
// magnifier 1/m folded in amp, micro-lens array); the Fresnel step is E_out = C E C^T (k_zgemm x 2).
// --------------------------------------------------------------------------------------
template <int ET>
static __global__ void k_sh_field_f64(const double* __restrict__ screens, const double* __restrict__ act,
                                      const double* __restrict__ modes, const double* __restrict__ aperture,
                                      const double* __restrict__ mla_phase, double2* __restrict__ E, int P, int Np,
                                      int K, int env0, int nB, int col_origin, double l_wfs, double amp) {
  extern __shared__ double sh_act[];   // [ET][K]
  const int e0 = blockIdx.y * ET;
  for (int i = threadIdx.x; i < ET * K; i += blockDim.x) {
    int e = i / K, k = i - e * K;
    sh_act[i] = (e0 + e < nB) ? act[(size_t)(env0 + e0 + e) * K + k] : 0.0;
  }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double s[ET];
#pragma unroll
  for (int e = 0; e < ET; ++e) s[e] = 0.0;
  for (int k = 0; k < K; ++k) {
    const double m = modes[(size_t)k * P + p];
#pragma unroll
    for (int e = 0; e < ET; ++e) s[e] = fma(m, sh_act[e * K + k], s[e]);
  }
  const double ap = aperture[p], ml = mla_phase[p];
  const int y = p / Np;
  int xp = p - y * Np + col_origin;
  if (xp >= Np) xp -= Np;
  const double kw = 6.283185307179586476925286766559 / l_wfs;
#pragma unroll
  for (int e = 0; e < ET; ++e)
    if (e0 + e < nB) {
      const double S = screens[(size_t)(env0 + e0 + e) * P + (size_t)xp * Np + y];
      double sn, cs;
      sincos(S / l_wfs + 2.0 * s[e] * kw + ml, &sn, &cs);
      E[(size_t)(e0 + e) * P + p] = make_double2(amp * ap * cs, amp * ap * sn);
    }
}

// The same field, folded by parity for a centrosymmetric Fresnel operator.  Thread = one pixel (i, x) of the
// top-left quadrant for ET envs; it forms the field at the four mirror-image pixels and writes
//   E_pq[i][x] = E[i][x] + p E[N-1-i][x] + q E[i][N-1-x] + p q E[N-1-i][N-1-x],   p, q = +-1
// as four [N/2][N/2] blocks: Efold[(p < 0) * 2 + (q < 0)][env][i * N/2 + x] (block stride = blk_stride elements).
template <int ET>
static __global__ void k_sh_field_fold(const double* __restrict__ screens, const double* __restrict__ act,
                                       const double* __restrict__ modes, const double* __restrict__ aperture,
                                       const double* __restrict__ mla_phase, double2* __restrict__ Efold,
                                       long long blk_stride, int P, int Np, int K, int env0, int nB, int col_origin,
                                       double l_wfs, double amp) {
  extern __shared__ double sh_act[];   // [ET][K]
  const int e0 = blockIdx.y * ET;
  for (int i = threadIdx.x; i < ET * K; i += blockDim.x) {
    int e = i / K, k = i - e * K;
    sh_act[i] = (e0 + e < nB) ? act[(size_t)(env0 + e0 + e) * K + k] : 0.0;
  }
  __syncthreads();
  const int Nh = Np / 2;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Nh * Nh) return;
  const int i = q / Nh, x = q - i * Nh;
  const int pix[4] = {i * Np + x, (Np - 1 - i) * Np + x, i * Np + (Np - 1 - x), (Np - 1 - i) * Np + (Np - 1 - x)};
  double s[4][ET];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int e = 0; e < ET; ++e) s[c][e] = 0.0;
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const double m = modes[(size_t)k * P + pix[c]];
#pragma unroll
      for (int e = 0; e < ET; ++e) s[c][e] = fma(m, sh_act[e * K + k], s[c][e]);
    }
  }
  const double kw = 6.283185307179586476925286766559 / l_wfs;
#pragma unroll
  for (int e = 0; e < ET; ++e)
    if (e0 + e < nB) {
      double2 E[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int y = pix[c] / Np;
        int xp = pix[c] - y * Np + col_origin;
        if (xp >= Np) xp -= Np;
        const double S = screens[(size_t)(env0 + e0 + e) * P + (size_t)xp * Np + y];
        const double ap = aperture[pix[c]];
        double sn, cs;
        sincos(S / l_wfs + 2.0 * s[c][e] * kw + mla_phase[pix[c]], &sn, &cs);
        E[c] = make_double2(amp * ap * cs, amp * ap * sn);
      }
      // c: 0 = (i, x), 1 = row-mirrored, 2 = column-mirrored, 3 = both
      const size_t o = (size_t)(e0 + e) * Nh * Nh + q;
      Efold[o] = make_double2(E[0].x + E[1].x + E[2].x + E[3].x, E[0].y + E[1].y + E[2].y + E[3].y);                       // p+ q+
      Efold[o + blk_stride] = make_double2(E[0].x + E[1].x - E[2].x - E[3].x, E[0].y + E[1].y - E[2].y - E[3].y);          // p+ q-
      Efold[o + 2 * blk_stride] = make_double2(E[0].x - E[1].x + E[2].x - E[3].x, E[0].y - E[1].y + E[2].y - E[3].y);      // p- q+
      Efold[o + 3 * blk_stride] = make_double2(E[0].x - E[1].x - E[2].x + E[3].x, E[0].y - E[1].y - E[2].y + E[3].y);      // p- q-
    }
}

// G_pq = C_p E_pq C_q^T (four [N/2][N/2] blocks per env) -> the full field: F at the four mirror images of (i, u) is
// the sum of the blocks weighted by 1, p, q, p q.
static __global__ void k_sh_unfold(const double2* __restrict__ G, long long blk_stride, double2* __restrict__ F, int Np,
                                   int nB) {
  const int Nh = Np / 2;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = blockIdx.y;
  if (q >= Nh * Nh || e >= nB) return;
  const int i = q / Nh, u = q - i * Nh;
  const size_t o = (size_t)e * Nh * Nh + q;
  const double2 a = G[o], b = G[o + blk_stride], c = G[o + 2 * blk_stride], d = G[o + 3 * blk_stride];
  double2* f = F + (size_t)e * Np * Np;
  f[(size_t)i * Np + u] = make_double2(a.x + b.x + c.x + d.x, a.y + b.y + c.y + d.y);
  f[(size_t)(Np - 1 - i) * Np + u] = make_double2(a.x + b.x - c.x - d.x, a.y + b.y - c.y - d.y);               // x p
  f[(size_t)i * Np + (Np - 1 - u)] = make_double2(a.x - b.x + c.x - d.x, a.y - b.y + c.y - d.y);               // x q
  f[(size_t)(Np - 1 - i) * Np + (Np - 1 - u)] = make_double2(a.x - b.x - c.x + d.x, a.y - b.y - c.y + d.y);    // x p q
}

// Photon noise of the Shack-Hartmann camera (hcipy large_poisson -> np.random.poisson, AO_env.py:274): an exact
// Poisson sampler on a Philox stream.  lambda < 10: Knuth's product of uniforms; lambda >= 10: Hoermann's transformed
// rejection with squeeze (PTRS, the algorithm NumPy itself uses; 86 % of draws accepted on the first uniform pair
// without a logarithm).  cuRAND's curand_poisson spends most of its time in the incomplete-gamma rejection of its
// 64 <= lambda < 4000 branch, which is where the lenslet pixels off the focal spot sit.
__device__ __forceinline__ double poisson_draw(curandStatePhilox4_32_10_t* st, double lam) {
  if (lam < 10.0) {
    if (lam <= 0.0) return 0.0;
    const double enlam = exp(-lam);
    double prod = 1.0;
    int k = 0;
    while (true) {
      prod *= curand_uniform_double(st);
      if (prod > enlam) ++k; else return (double)k;
    }
  }
  const double slam = sqrt(lam), loglam = log(lam);
  const double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
  const double invalpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
  while (true) {
    const double U = curand_uniform_double(st) - 0.5, V = curand_uniform_double(st);
    const double us = 0.5 - fabs(U);
    const double k = floor((2.0 * a / us + b) * U + lam + 0.43);
    if (us >= 0.07 && V <= vr) return k;
    if (k < 0.0 || (us < 0.013 && V > us)) continue;
    if (log(V) + log(invalpha) - log(a / (us * us) + b) <= -lam + k * loglam - lgamma(k + 1.0)) return k;
  }
}

// test hook (aog_debug_poisson): n draws at one rate, one Philox subsequence per draw as the camera kernel uses them
static __global__ void k_debug_poisson(double lam, int n, unsigned long long seed, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  curandStatePhilox4_32_10_t st;
  curand_init(seed, (unsigned long long)i, 0ull, &st);
  out[i] = (lam > 1e6) ? rint(lam + sqrt(lam) * curand_normal_double(&st)) : poisson_draw(&st, lam);
}

// camera image (power x dt), photon noise, flux-weighted centroids per selected lenslet (one warp each,
// deterministic), slopes, leaky integrator a <- 0.99 a - 0.3 R slopes.  Block per env.
static __global__ void k_sh_centroid_update(const double2* __restrict__ F, long long strideF,
                                            const int* __restrict__ off, const int* __restrict__ pix,
                                            const double* __restrict__ px, const double* __restrict__ py,
                                            const double* __restrict__ offset, const double* __restrict__ recon,
                                            double* __restrict__ act_sh, double* __restrict__ action_out,
                                            const double* __restrict__ noisy, int P, int K, int Nsub, int env0,
                                            double weight_dt, int noise_mode, unsigned long long seed,
                                            unsigned long long env_id_base, unsigned long long draw) {
  extern __shared__ double slopes[];   // [2 Nsub]
  const int b = blockIdx.x;
  const double2* f = F + (size_t)b * strideF;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int m = warp; m < Nsub; m += nw) {
    double fl = 0.0, sx = 0.0, sy = 0.0;
    for (int i = off[m] + lane; i < off[m + 1]; i += 32) {
      const int p = pix[i];
      double v;
      if (noise_mode == AOG_SH_NOISE_INJECTED) {
        v = noisy[(size_t)(env0 + b) * P + p];
      } else {
        const double2 e = f[p];
        v = (e.x * e.x + e.y * e.y) * weight_dt;
        if (noise_mode == AOG_SH_NOISE_POISSON) {     // hcipy large_poisson: Poisson below 1e6, rounded normal above
          curandStatePhilox4_32_10_t st;
          // one Philox subsequence per (global env, pixel); successive SH_step draws are 256 outputs apart
          curand_init(seed, (env_id_base + env0 + b) * (unsigned long long)P + p, draw * 256ull, &st);
          v = (v > 1e6) ? rint(v + sqrt(v) * curand_normal_double(&st)) : poisson_draw(&st, v);
        }
      }
      v += 1e-10;                                     // AO_env.py:277
      fl += v; sx += v * px[i]; sy += v * py[i];
    }
    fl = warp_sum(fl); sx = warp_sum(sx); sy = warp_sum(sy);
    if (lane == 0) {
      slopes[m] = sx / fl - offset[m];
      slopes[Nsub + m] = sy / fl - offset[Nsub + m];
    }
  }
  __syncthreads();
  // a <- 0.99 a - 0.3 R slopes: one warp per reconstructor row, lanes along the row (coalesced), fixed-order tree sum
  for (int k = warp; k < K; k += nw) {
    double r = 0.0;
    for (int m = lane; m < 2 * Nsub; m += 32) r += recon[(size_t)k * 2 * Nsub + m] * slopes[m];
    r = warp_sum(r);
    if (lane == 0) {
      const size_t i = (size_t)(env0 + b) * K + k;
      const double a = (1.0 - 0.01) * act_sh[i] - 0.3 * r;
      act_sh[i] = a;
      if (action_out) action_out[i] = a;
    }
  }
}

static __global__ void k_broadcast_rows(const double* __restrict__ row, double* __restrict__ out, int K, int B) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K * B) out[i] = row[i % K];
}

// misc ---------------------------------------------------------------------------------
// caller's screens [count][y][x] (row-major, as hcipy's Field) -> device screens [count][x][y] FP64
template <typename T>
static __global__ void k_screens_in(const T* __restrict__ in, double* __restrict__ out, int Np, size_t n) {
  const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n) return;
  const size_t P = (size_t)Np * Np, b = o / P, r = o - b * P;
  const int x = (int)(r / Np), y = (int)(r - (size_t)x * Np);
  out[o] = (double)in[b * P + (size_t)y * Np + x];
}

static __global__ void k_transpose_z(const double2* __restrict__ in, double2* __restrict__ out, int rows, int cols) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) { int r = i / cols, c = i - r * cols; out[(size_t)c * rows + r] = in[i]; }
}

static __global__ void k_build_arW(const double* __restrict__ A, const double* __restrict__ Bm, const int* __restrict__ perm,
                            double* __restrict__ W, int Np, int Ns, int reverse_cols) {
  // W[j][y] = A[y][perm[j]] (j < Ns: stencil point j of the gather order);  W[Ns + j][y] = B[y][j]
  // reverse_cols: the rows of the two full stencil columns in reversed order (k_ar_step<DIRECT> on the rotated screen)
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (Ns + Np) * Np) return;
  int j = i / Np, y = i - j * Np;
  int js = j;
  if (reverse_cols && j < 2 * Np) js = (j / Np) * Np + (Np - 1 - j % Np);
  W[i] = (j < Ns) ? A[(size_t)y * Ns + perm[js]] : Bm[(size_t)y * Np + (j - Ns)];
}
