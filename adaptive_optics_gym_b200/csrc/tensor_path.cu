// Tensor-core arithmetic of the AO-v0 step path (AOG_PRECISION_FUSED and AOG_PRECISION_TENSOR), sm_100a only.
//
// AOG_PRECISION_FUSED -- one optics kernel per chunk of environments:
//   k_actuators_pack  action -> normalised actuators -> split-fp16 GEMM operand
//   k_dm_phase_tc<.., MODE 1 | 2>  DM surface as a tcgen05 GEMM over blocks of 128 envs; epilogue = total wavefront
//                   phase (atmosphere + DM) and, from it, every output of the step as sums over the pupil: obs-arm
//                   column sums, Strehl sum, fibre-coupling coefficients as inner products with the fibre modes
//                   propagated back to the pupil (G_j = M1^T (mode_j w) M2^T).  Nothing but partial sums leaves the SM.
//   k_small_fused   the same optics chain with a thread per pixel for batches of at most 8 envs (one env = configs[0])
//   k_finalize_tcw  detector powers, fibre power, Strehl, SSIM, reward: one warp per env
//
// AOG_PRECISION_TENSOR -- the fibre arm through the matrix Fourier transform, three kernels per chunk:
//   k_dm_phase_tc   DM surface as a tcgen05 GEMM over blocks of 128 envs; epilogue = total wavefront phase
//                   (atmosphere + DM) -> HBM as FP32 radians, obs-arm column sums, Strehl sums
//   k_field_mft1    field warps turn that phase into the pupil field ON CHIP (sincos, aperture, fp16 hi/lo) as the
//                   B operand of the first matrix-Fourier-transform product; epilogue = stage-1 product, split fp16
//   k_mft2          second product with the fibre-mode projection in its epilogue
//
// The matrix Fourier transform F = M1 . E . M2 (reference AO_env.py:138 -> hcipy FraunhoferPropagator /
// MatrixFourierTransform) runs as two real-embedded complex GEMMs on the 5th-gen tensor cores (tcgen05.mma
// cta_group::2 kind::f16, M = 256 over a CTA pair, FP32 accumulators in TMEM), operands staged in shared memory
// by TMA (cp.async.bulk.tensor, SWIZZLE_64B) through mbarrier rings:
//
//   stage 1  [Tr ; Ti] (256 x 240) = [[M1r, -M1i], [M1i, M1r]] (256 x 480) . [Er ; Ei] (480 x 240)
//   stage 2  [Fr ; Fi]^T (256 x 256) = [[M2r, -M2i], [M2i, M2r]]^T (256 x 480) . [T(env a) | T(env b)] (480 x 256)
//
// Precision: every operand is split x = hi + lo into two fp16 values (|x| <= 240, so the pair carries ~22 bits) and
// each product is issued as hi.hi + hi.lo + lo.hi ("3x split"), which keeps FP32-class accuracy at fp16 tensor
// throughput.  The unit-modulus twiddle tables are split once on the host from their FP64 values; the pupil field is
// split by the field warps, the stage-1 product by the stage-1 epilogue.  The stage-2 epilogue never writes the focal
// plane: it projects it on the fibre modes (AO_env.py:471) out of TMEM.
#include "tensor_path.cuh"
#include "finalize.cuh"
#include "philox.cuh"
#include "fp32x2.cuh"
#include "phase_round.cuh"

#include <cuda.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <string>
#include <vector>

struct TensorState {
  // operands (device)
  DevArray<__half> A1_hi, A1_lo;                      // [256][480]  stage-1 constant
  DevArray<__half> B2_hi, B2_lo;                      // [256][480]  stage-2 constant (N-major rows, K contiguous)
  DevArray<__half> T_hi, T_lo;                        // [chunk][128][480]  stage-1 product
  DevArray<float> lpw;                                // [J][128][128] fibre modes * weight / max
  DevArray<float> lpwr;                               // the same, [rank][v / 16][J][(v / 4) % 4][64 u][4 v] (stage-2 epilogue tiles)
  DevArray<double> coef4;                             // [chunk][J][re|im][rank] raw projection sums
  // atmospheric phase at lambda_wfs, UNREDUCED, int32 fixed point in units of 2^-22 half-turns (PHI_ONE per
  // half-turn; +-512 half-turns of range), tiled for the phase kernel's bulk prefetch:
  // [env / 32][Np xp][Np / 16 chunks][32 envs][16 pixels], ring-buffered in xp, the four 16-byte pieces of
  // each env row pre-swizzled (piece j at j ^ ((env >> 1) & 3)) so the shared-memory image is conflict free.
  DevArray<int32_t> hwt;
  // the same tiles as a 5-D tensor [env / 32][Np xp][Np / 16][32][16]: one box = the four 32-env tiles of a 128-env
  // block at one (column, chunk), 8 KB, for the shared prefetch of the phase kernel's lane groups
  CUtensorMap tmHwt;
  // total wavefront phase (atmosphere + DM) at lambda_wfs reduced to [-pi, pi) radians, FP32,
  // [chunk][Np / 16 (y chunk)][Np x][16 y] (the 120 columns x 16 pixels one CTA needs per K block are one
  // contiguous 7.5 KB run): written by the phase kernel, read by the stage-1 kernel's field warps, which form
  // the pupil field on chip -- the field itself never goes to HBM.
  DevArray<float> phi;
  CUtensorMap tmPhi;
  DevArray<__half> modesK_hi, modesK_lo;              // [Np x][Np y][KPAD] DM modes, k contiguous (GEMM B operand)
  DevArray<__half> act_hi, act_lo;                    // [chunk rows padded to 128][KPAD] actuators * 4 / lambda_wfs
  DevArray<uint16_t> apmask;                          // [Np x][Np / 16] aperture bits of each 16-pixel column chunk
  DevArray<float2> R4;                                // [chunk][Np x][FK_PARTS][n] obs-arm column partial sums
  DevArray<float2> m1o32;                             // [n][Np] first obs-arm table in FP32
  int kpad = 64;
  int act_rows = 128;
  DevArray<double2> m2oT;                             // [n][Np] transposed obs table
  int* err_flag = nullptr;                            // not owned: device alias of err_flag_host, set by a timed-out barrier wait
  PinnedArray<int> err_flag_host;
  // AOG_PRECISION_FUSED: per-pixel records [Np x][Np / 16][16 y][FK_NT(n)] float2 = [obs-arm twiddles m1o[v][y] |
  // fibre modes propagated back to the pupil, G_j = M1^T (mode_j w) M2^T / max|G| | (aperture, 0)], all times the
  // aperture: the 16 records of a column chunk are one contiguous run for the bulk prefetch
  bool fused = false;
  bool packed_valid = false;                          // act_hi / act_lo already hold this step's actuators (k_actuators_pack)
  DevArray<float2> gfib;
  double gfib_scale = 0.0;
  DevArray<double2> fib_part;                         // [chunk][FK_SLOTS][FK_JT] partial projection sums
  bool have_gfib = false, have_G = false;
  std::vector<double> h_m1, h_m2, h_lp, h_G, h_m1o, h_ap;   // host copies of the tables the records are built from
  // symmetric tables (kernel MODE 2, see FK_NF): G_j = e^{i theta_j} R_j; lpphase_f[j] = e^{i beta_j L} e^{i theta_j}
  bool sym = false, g_real = false, have_lpphase = false;
  double theta[AOG_MAX_LP] = {0};
  std::vector<double> h_lpphase;
  DevArray<double2> lpphase_f;
  CUtensorMap tmA1_hi, tmA1_lo, tmB2_hi, tmB2_lo;
  CUtensorMap tmT128_hi, tmT128_lo;
  CUtensorMap tmTout_hi, tmTout_lo;                   // stage-1 epilogue stores: 128 rows x 16 columns, SWIZZLE_32B                   // stage-1 product, one env (128 rows) per box
  CUtensorMap tmAct_hi, tmAct_lo, tmModes_hi, tmModes_lo;
  // ---- Shack-Hartmann integrator on the tensor cores (sh_tensor.cuh) ----
  std::vector<double> h_shC, h_shMla, h_shPx, h_shPy;  // host copies of the SH tables the operands are built from
  std::vector<int> h_shOff, h_shPix;
  bool sh_have[6] = {false, false, false, false, false, false};   // fresnel, mla, offsets, index, x, y
  bool sh_ready = false, sh_unsupported = false;
  std::string sh_why;                                 // why the tables do not qualify (the FP64 kernels run instead)
  DevArray<__half> shCE_hi[2];                        // [stage][2 parities][re | im][128 rows][256 K] operator embeddings
  DevArray<__half> shCE_lo[2];
  DevArray<__half> shEB_hi, shEB_lo;                  // [chunk][p][q][128 x][256 K] folded field
  DevArray<__half> shYB_hi, shYB_lo;                  // [chunk][q][p][128 i'][256 K] first product
  DevArray<float> shG;                                // [chunk][p][q][128 i'][re 128 | im 128] second product
  DevArray<int16_t> shSlot;                           // [P] lenslet slot of each camera pixel
  DevArray<double> shSlotC;                           // [Nsub][3]
  double shScale[2] = {1.0, 1.0};                     // power-of-two scales of the two operator tables
  double shX0 = 0, shdX = 0, shY0 = 0, shdY = 0;
  CUtensorMap tmShCE_hi[2], tmShCE_lo[2], tmShEB_hi, tmShEB_lo, tmShYB_hi, tmShYB_lo, tmShYout_hi, tmShYout_lo;
  bool sh_buffers = false;
  double pupil_weight = 0.0;                          // |M1| (grid weight folded in the table)
  double lpw_scale = 0.0;
  int num_sms = 148;
  bool have_m1 = false, have_m2 = false, have_lp = false, have_modes = false, have_ap = false, have_m2o = false, have_m1o = false;
};

void TensorStateDeleter::operator()(TensorState* ts) const { delete ts; }

namespace {

constexpr int TC_NP = 240;          // pupil pixels per side this path is built for
constexpr int TC_NF = 128;          // focal pixels per side
constexpr int TC_K = 2 * TC_NP;     // real-embedded contraction length (480)
constexpr int KB = 32;              // K elements per pipeline stage (64 B rows, SWIZZLE_64B)
constexpr int NUM_KB = TC_K / KB;   // 15
constexpr int A_TILE = 128 * KB * 2;            // 8 KB: 128 rows x 64 B
constexpr float PHI_ONE = 4194304.f;   // 2^22 fixed-point units per half-turn of phase

// ----------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (the launch fails, the GPU stays usable), never hang.
template <int SLEEP_NS = 0>
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err_flag, int code) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
    if (++spins > (1u << 24)) {            // seconds: a protocol bug, not a slow producer
      *(volatile int*)err_flag = code;          // mapped host memory: a plain store, then a system-scope fence
      __threadfence_system();
      asm volatile("trap;");
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): rows of 64 B,
// 8-row groups 512 B apart (SBO), LBO = 1 (ignored for swizzled K-major), version 1 (Blackwell).
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;   // LayoutType::SWIZZLE_64B
  return d;
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = F16, K-major both.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ----------------------------------------------------------------------------- the GEMM kernel
__device__ __forceinline__ void split_pack2(float a, float b, uint32_t& hi, uint32_t& lo);

struct TcParams {
  int num_items;        // MODE 0: envs;  MODE 1: env pairs
  int num_envs;         // envs in this chunk
  // MODE 0 epilogue: stage-1 product as split fp16, [env][128][480]
  __half* T_hi; __half* T_lo;
  // MODE 1 epilogue: fibre projection, raw sums [env][J][2] (re from cluster rank 0, im from rank 1)
  const float* lpw;     // [J][128][128]
  const float* lpwr;    // same weights as [rank 2][v / 16][J][(v / 4) % 4][64 u][4 v]: one contiguous tile per (rank, 16 rows)
  double* coef_raw;     // [env][J][part re|im][rank] partial projection sums
  int J;
  int dbg;              // AOG_TC_DEBUG bits (tuning experiments only): 1 no MMA, 2 no TMA, 4 no epilogue work
  int* err_flag;
};

// ----------------------------------------------------------------------------- MFT stage 2 (pair MMA)
// k_mft2: the second MFT product with the fibre projection in its epilogue, as cta_group::2 MMAs (M = 256 over the
// CTA pair; each CTA holds 128 rows of A and HALF of the B tile in its own shared memory, so no operand is
// multicast or duplicated).  item = env pair; computes F^T:
//   A = twiddle rows (CTA 0: Fr, CTA 1: Fi; M = focal column u), B = the stage-1 products of the two envs
//   stacked along N = 2 x 128 focal rows v (CTA r stages env 2 item + r), K = 480 = (x | 240 + x).
// Only the leader CTA (rank 0) issues MMAs; both CTAs' TMA loads complete on the leader's `full` barrier,
// tcgen05.commit multicasts `empty` / `tmem_full` to both CTAs, and both CTAs' epilogue warps arrive on the
// leader's `tmem_empty`.  8 epilogue warps per CTA (two per TMEM lane group, half of the columns each).
// TMEM holds SEPARATE accumulators for the main hi.hi chain and for the hi.lo + lo.hi corrections: the tensor
// core truncates its FP32 accumulation, so every accumulate onto a large sum costs ~ -0.5 ulp; keeping the
// 2 x 30 tiny correction updates off the main accumulator cuts that bias 3x (tools/tensor_bias_probe.py).
constexpr int M2_STAGES = 5;
constexpr int M2_STAGE_BYTES = 4 * A_TILE;          // 32 KB: [A_hi][A_lo][B_hi slot][B_lo slot], 8 KB each
constexpr int M2_EPI_WARPS = 8;
constexpr int M2_THREADS = (3 + M2_EPI_WARPS) * 32; // 352: TMA, MMA, 8 epilogue, fibre-weight loader
constexpr int M2_OUT_TILE = 128 * 16 * 2;           // stage-1 kernel: 4 KB, 128 rows x 16 fp16 of its product (SWIZZLE_32B)
constexpr int M2_OUT_BUFS = 3;                      // stage-1 kernel: per column half, ring of (hi, lo) tile pairs for the TMA stores
constexpr int M2_EPI_BYTES = 2 * M2_OUT_BUFS * 2 * M2_OUT_TILE;   // 48 KB
constexpr int M2_SMEM_BYTES = M2_STAGES * M2_STAGE_BYTES + 4 * 3 * 4096 /*fibre-weight ring*/ + 1024 /*align*/ + 4096 /*barriers + reduction scratch*/;

__device__ __forceinline__ uint32_t mapa_rank(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// TMA load whose completion is signalled on a barrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr,
                                                 int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// Arrive on a barrier that may live in the peer CTA.  CTA-scope release (the PTX default, as CUTLASS's
// ClusterBarrier::arrive): what is handed over lives in shared memory and is published to the async proxy by the
// caller's fence.proxy.async; a cluster-scope release here would also wait for the caller's outstanding global
// loads (the phase prefetch) and flush L1 on every K block.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// JT: compile-time bound on the fibre modes held in registers (3 = the reference's LP01 + 2 x LP11; 8 = generic).
// Row split: CTA r owns the focal columns u in [64 r, 64 r + 64) for BOTH parts of F^T -- its A rows are
// [Fr rows of those u | Fi rows of those u] (TMEM lanes 0-63 | 64-127) -- so the real fibre weights of a
// (u, v) are shared by the Fr and Fi lanes and each CTA streams half of the weight table: per 16 focal rows v
// one contiguous tile [j][v / 4][64 u][4 v] (4 KB per mode), fetched by a dedicated warp with cp.async.bulk
// into a 4-slot ring (JT <= 3) and read conflict-free (lane = u).  Epilogue warp (lane group lg, env e):
// part = lg / 2 (Fr | Fi), all 128 focal rows v of env e.
constexpr int M2_W_SLOTS = 4;
constexpr int M2_W_SLOT_BYTES = 3 * 4096;                            // up to 3 modes x [4][64][4] floats
template <int JT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(M2_THREADS, 1)
k_mft2(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
       const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo, const TcParams p) {
  constexpr int N_MMA = 2 * TC_NF;                                   // 256
  constexpr int B_ROWS = N_MMA / 2;                                  // rows of B each CTA stages: 128
  constexpr bool W_RING = JT <= 3;
  // bytes landing per stage over BOTH CTAs (all of them complete on the leader's barrier)
  constexpr uint32_t TX_BYTES = 2 * (2 * A_TILE + 2 * B_ROWS * KB * 2);
  constexpr uint32_t IDESC = umma_idesc_f16(256, N_MMA);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* wring = base + M2_STAGES * M2_STAGE_BYTES;                // fibre-weight tile ring
  uint64_t* full = reinterpret_cast<uint64_t*>(wring + M2_W_SLOTS * M2_W_SLOT_BYTES);
  uint64_t* empty = full + M2_STAGES;
  uint64_t* w_full = empty + M2_STAGES;
  uint64_t* w_empty = w_full + M2_W_SLOTS;
  uint64_t* tmem_full = w_empty + M2_W_SLOTS;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  double* red = reinterpret_cast<double*>(wring + M2_W_SLOTS * M2_W_SLOT_BYTES + 256);   // [2 bufs][8 warps][AOG_MAX_LP]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_lo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB_lo)) : "memory");
    for (int s = 0; s < M2_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < M2_W_SLOTS; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], M2_EPI_WARPS); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 2 * M2_EPI_WARPS);          // every epilogue warp of both CTAs (used in the leader only)
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs; completion on the leader's barrier) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        const int b_row0 = (2 * item + (int)rank) * TC_NF;
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait<32>(&empty[stage], phase ^ 1, p.err_flag, 1);
          if (p.dbg & 2) { if (rank == 0) mbar_arrive(&full[stage]); if (++stage == M2_STAGES) { stage = 0; phase ^= 1; } continue; }
          if (rank == 0) mbar_expect_tx(&full[stage], TX_BYTES);
          const uint32_t s0 = smem_u32(base + stage * M2_STAGE_BYTES);
          const uint32_t fb = mapa_rank(smem_u32(&full[stage]), 0);
          const int k0 = kb * KB;
          tma_load_2d_pair(s0, &tmA_hi, fb, k0, (int)rank * 128);
          tma_load_2d_pair(s0 + A_TILE, &tmA_lo, fb, k0, (int)rank * 128);
          tma_load_2d_pair(s0 + 2 * A_TILE, &tmB_hi, fb, k0, b_row0);
          tma_load_2d_pair(s0 + 3 * A_TILE, &tmB_lo, fb, k0, b_row0);
          if (++stage == M2_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread of the leader CTA) =====================
    if (rank == 0 && lane == 0) {
      int stage = 0;
      uint32_t phase = 0, tphase = 0;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        mbar_wait<32>(tmem_empty, tphase ^ 1, p.err_flag, 2);
        tc_fence_after();
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait(&full[stage], phase, p.err_flag, 3);
          tc_fence_after();
          const uint32_t s0 = smem_u32(base + stage * M2_STAGE_BYTES);
          if (!(p.dbg & 1))
#pragma unroll
          for (int ks = 0; ks < KB / 16; ++ks) {
            const uint32_t acc = (kb | ks) != 0;
            const uint64_t a_hi = umma_desc_sw64(s0 + ks * 32), a_lo = umma_desc_sw64(s0 + A_TILE + ks * 32);
            const uint64_t b_hi = umma_desc_sw64(s0 + 2 * A_TILE + ks * 32);
            const uint64_t b_lo = umma_desc_sw64(s0 + 3 * A_TILE + ks * 32);
            tc_mma_f16_pair(tmem_base, a_hi, b_hi, IDESC, acc);              // main
            tc_mma_f16_pair(tmem_base + 256, a_hi, b_lo, IDESC, acc);        // corrections
            tc_mma_f16_pair(tmem_base + 256, a_lo, b_hi, IDESC, 1);
          }
          tc_commit_pair(&empty[stage]);            // frees the slot in both CTAs when these MMAs retire
          if (++stage == M2_STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_pair(tmem_full);
        tphase ^= 1;
      }
    }
  } else if (warp == 2 + M2_EPI_WARPS) {
    // ===================== fibre-weight tiles: the same 8 tiles for every env pair =====================
    if (W_RING && lane == 0 && !(p.dbg & 4)) {
      int slot = 0;
      uint32_t phase = 0;
      const uint32_t bytes = (uint32_t)p.J * 4096u;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        for (int c = 0; c < TC_NF / 16; ++c) {
          mbar_wait<64>(&w_empty[slot], phase ^ 1, p.err_flag, 9);
          mbar_expect_tx(&w_full[slot], bytes);
          const float* src = p.lpwr + ((size_t)((int)rank * (TC_NF / 16) + c) * p.J) * 1024;
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(smem_u32(wring + slot * M2_W_SLOT_BYTES)), "l"(src), "r"(bytes), "r"(smem_u32(&w_full[slot])) : "memory");
          if (++slot == M2_W_SLOTS) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue: 8 warps, TMEM lane group = warp % 4, env of the pair = (warp - 2) / 4 ========
    const int lg = warp & 3;
    const int e = (warp - 2) >> 2;
    const int row = lg * 32 + lane;
    const int ul = row & 63;                           // focal column within my CTA's 64
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
    const uint32_t tmem_empty_leader = mapa_rank(smem_u32(tmem_empty), 0);
    uint32_t tphase = 0, wphase = 0;
    int wslot = 0;
    int it = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters, ++it) {
      mbar_wait(tmem_full, tphase, p.err_flag, 4);
      tc_fence_after();
      tphase ^= 1;
      if (p.dbg & 4) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tmem_empty_leader);
        continue;
      }
      // Phase 1: drain env e's 128 columns (main + corrections) into registers and hand the TMEM back.
      float f[128];
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        float a[32], b[32];
        tc_ld32(lane_addr + e * 128 + c * 16, a);
        tc_ld32(lane_addr + 256 + e * 128 + c * 16, b);
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 32; ++q) f[c * 16 + q] = a[q] + b[q];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty_leader);   // TMEM is free: the next pair's MMAs may start
      // Phase 2: fibre projection of my part (Fr | Fi) of my 64 focal columns: FP32 per 16 rows, FP64 across.
      double acc[JT];
#pragma unroll
      for (int j = 0; j < JT; ++j) acc[j] = 0.0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float s[JT];
#pragma unroll
        for (int j = 0; j < JT; ++j) s[j] = 0.f;
        if constexpr (W_RING) {
          mbar_wait(&w_full[wslot], wphase, p.err_flag, 10);
          const float4* wt = reinterpret_cast<const float4*>(wring + wslot * M2_W_SLOT_BYTES) + ul;
#pragma unroll
          for (int j = 0; j < JT; ++j)
            if (j < p.J) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 w = wt[(j * 4 + q) * 64];
                s[j] = fmaf(f[c * 16 + 4 * q + 0], w.x, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 1], w.y, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 2], w.z, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 3], w.w, s[j]);
              }
            }
          __syncwarp();
          if (lane == 0) mbar_arrive(&w_empty[wslot]);
          if (++wslot == M2_W_SLOTS) { wslot = 0; wphase ^= 1; }
        } else {
          const float4* wt = reinterpret_cast<const float4*>(p.lpwr) + ((size_t)((int)rank * (TC_NF / 16) + c) * p.J) * 256 + ul;
#pragma unroll
          for (int j = 0; j < JT; ++j)
            if (j < p.J) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 w = __ldg(wt + (j * 4 + q) * 64);
                s[j] = fmaf(f[c * 16 + 4 * q + 0], w.x, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 1], w.y, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 2], w.z, s[j]);
                s[j] = fmaf(f[c * 16 + 4 * q + 3], w.w, s[j]);
              }
            }
        }
#pragma unroll
        for (int j = 0; j < JT; ++j) acc[j] += (double)s[j];
      }
      double* rbuf = red + (it & 1) * (M2_EPI_WARPS * AOG_MAX_LP);
      const int ew = warp - 2;                          // = e * 4 + lg
#pragma unroll
      for (int j = 0; j < JT; ++j)
        if (j < p.J) {
          const double a = warp_sum(acc[j]);
          if (lane == 0) rbuf[ew * AOG_MAX_LP + j] = a;
        }
      asm volatile("bar.sync 1, %0;" ::"n"(M2_EPI_WARPS * 32) : "memory");
      if (warp == 2 && lane < 4 * p.J) {
        // (env of the pair, part, mode): sum of the two lane groups of that part
        const int j = lane % p.J, pe = lane / p.J, part = pe & 1, ee = pe >> 1;
        const int env = 2 * item + ee;
        if (env < p.num_envs)
          p.coef_raw[(((size_t)env * p.J + j) * 2 + part) * 2 + rank] =
              rbuf[(ee * 4 + 2 * part) * AOG_MAX_LP + j] + rbuf[(ee * 4 + 2 * part + 1) * AOG_MAX_LP + j];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  // neither CTA may exit (or free its TMEM) while the pair's MMAs, loads or barrier signals can still touch it
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ----------------------------------------------------------------------------- phase kernel
// k_dm_phase_tc: DM surface as a tensor-core GEMM with the wavefront-phase formation in its epilogue
// (reference AO_env.py:119-120 surface, :132-135 atmosphere + DM phase, :479-483 Strehl sum).
//
//   D[env][y] (half-turns of DM phase at lambda_wfs) = act'[env][k] . modes[x][y][k]      per pupil column x
//
// A = 128 envs x KPAD (actuators scaled by 4 / lambda_wfs, split fp16), B = the 240 pixels of column x
// (split fp16 modes, k contiguous), accumulator = 128 TMEM lanes (envs) x 240 columns (pixels), double
// buffered (2 x 256 columns).  12 epilogue warps (3 per TMEM lane group, each a third of the column)
// own ONE ENV PER THREAD: add the atmospheric phase (int32 fixed point, bulk-prefetched tiles), store the
// total phase (reduced, FP32 radians) for the stage-1 kernel's field warps, and accumulate in registers the
// obs-arm column sums R[x][v] = sum_y m1o[v][y] E[y][x] (AO_env.py:139; FP32 per 16 pixels, FP64 across)
// and the Strehl sum sum_ap exp(i phi lambda_wfs / lambda_sci).
// Work item = (block of 128 envs, column x, segment s); each CTA takes a contiguous range of items.  A pupil column
// longer than 256 pixels (NP = 512) is split into NSEG = 2 segments of SEG = 256 pixels, one MMA (N = SEG) each: the
// N of one MMA, a TMA box and one half of the double-buffered accumulator all stop at 256.
constexpr int FK_STAGES = 1;                            // the double-buffered TMEM accumulator hides the operand load
constexpr int FK_A_TILE = 128 * 64 * 2;                 // 16 KB: 128 env rows x 128 B
constexpr int FK_B_TILE = 256 * 64 * 2;                 // 32 KB slot (240 rows used)
__host__ __device__ constexpr int FK_NSEG(int np) { return np > 256 ? 2 : 1; }
constexpr int FK_STAGE_BYTES = 2 * FK_A_TILE + 2 * FK_B_TILE;   // 96 KB
#ifndef AOG_FK_EPI_WARPS      // tuning builds: 12 or 16
#define AOG_FK_EPI_WARPS 12
#endif
constexpr int FK_EPI_WARPS = AOG_FK_EPI_WARPS;          // 3 per TMEM lane group: 5 of the 15 column chunks each
constexpr int FK_PARTS = FK_EPI_WARPS / 4;
// Work item -> column segment xs = x NSEG + s: a CTA's contiguous item range strides through the pupil (53 is coprime
// with 240 and 1024), so every CTA sees the same mix of short (edge) and long (centre) aperture chords.
// (The tensor path's phase kernel keeps the natural order: its phase stores of neighbouring columns are neighbours
// in HBM, and striding them costs more DRAM page misses than the imbalance does.)
constexpr int FK_COL_STRIDE = 53;
template <int MODE, int NP>
__device__ __forceinline__ int fk_segment(int item_in_block) {
  // 53 is prime: coprime with every NP NSEG
  return (MODE == 0 || MODE == 3) ? item_in_block : (item_in_block * FK_COL_STRIDE) % (NP * FK_NSEG(NP));
}
constexpr int FK_THREADS = (2 + FK_EPI_WARPS) * 32;     // 448

constexpr int FK_SLOTS = 128;                           // Strehl / fibre partial slots per env (>= CTAs touching an env block)
constexpr int FK_MIN_ITEMS = 2;                         // items per CTA at least (with a bound from FK_SLOTS); small batches spread over more SMs
constexpr int FK_PF_TILE = 32 * 16 * 4;                 // 2 KB: 32 envs x 16 pixels of phase (one bulk copy)
constexpr int FK_JT = 3;                                // fibre modes of the fused kernel (LP01 + 2 x LP11, AO_env.py:393)
// Fused kernel: per pixel one record of FK_NT(n) float2 = [n obs-arm twiddles | FK_JT back-projected fibre modes |
// (aperture, 0)], every entry already multiplied by the aperture, so the arithmetic needs no mask; the 16 records
// of a (column, 16-pixel chunk) are one contiguous run fetched with the phase tile.
__host__ __device__ constexpr int FK_NT(int nobs) { return (nobs + FK_JT + 1 + 1) & ~1; }
// Symmetric fused kernel (kernel MODE 2).  hcipy's pupil and focal grids are symmetric about the axis, so
//   * the obs-arm twiddle rows come in conjugate pairs, m1o[n-1-v][y] = conj(m1o[v][y]) (the centre row of an odd n
//     is real): with m = a + ib and E = c + is the four products ac, bs, as, bc serve both rows of a pair;
//   * every back-projected fibre mode is a real function times one unit phasor, G_j = e^{i theta_j} R_j (the Fourier
//     transform of a real mode that is even or odd along each axis): the projection is two real sums and the phasor
//     joins the mode's propagation phase in k_finalize_tcw.
// Record = FK_NF(n) floats: [a, b per pair | centre a | R_0..R_2 | aperture], padded to a multiple of 4.
// The tables are checked for both properties when they are uploaded; tables without them run kernel MODE 1.
__host__ __device__ constexpr int FK_NF(int nobs) { return (2 * (nobs / 2) + (nobs & 1) + FK_JT + 1 + 3) & ~3; }
// kernel MODE: 0 = tensor path (stores the phase for the MFT stages), 1 = fused, 2 = fused + symmetric tables,
// 3 = phase only (the Shack-Hartmann path, sh_tensor.cuh: stores the phase, no detector / Strehl sums)
__host__ __device__ constexpr int FK_TAB_TILE(int nobs, int mode) {
  return mode == 1 ? 16 * FK_NT(nobs) * 8 : (mode == 2 ? 16 * FK_NF(nobs) * 4 : 0);
}
// Prefetch ring of one q group (the four warps, one per TMEM lane group, that walk the same chunk stream): a slot
// holds one chunk's four 2 KB phase tiles (lane group lg at lg x 2 KB, one tensor copy) and its one record tile.
constexpr int FK_PF_STAGES = 3;
constexpr int FK_PF_PHASE = 4 * FK_PF_TILE;             // 8 KB
__host__ __device__ constexpr int FK_PF_SLOT(int nobs, int mode) { return (FK_PF_PHASE + FK_TAB_TILE(nobs, mode) + 127) & ~127; }
__host__ __device__ constexpr int FK_PF_BYTES(int nobs, int mode) { return FK_PARTS * FK_PF_STAGES * FK_PF_SLOT(nobs, mode); }
constexpr int FK_AUX_BAR = 512;

__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;   // 8 rows x 128 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;             // LayoutType::SWIZZLE_128B
  return d;
}

// sin / cos of a fixed-point phase (PHI_ONE units per half-turn): the low 23 bits are the phase mod one turn,
// exactly; the SFU (MUFU.SIN / MUFU.COS) has abs error 2^-21.4 on [-pi, pi].
// int -> float for |v| < 2^22 without the conversion (XU) pipe: 1.5 * 2^23 + v is exact in FP32
__device__ __forceinline__ float small_int_to_float(int32_t v) {
  return __int_as_float(v + 0x4B400000) - 12582912.f;
}
__device__ __forceinline__ void sincos_fixed(int32_t t, float* s, float* c) {
  const float x = small_int_to_float((t << 9) >> 9) * (3.14159265358979323846f / PHI_ONE);
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(*s) : "f"(x));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(*c) : "f"(x));
}

// sin / cos of a fixed-point phase given as tb = t + 2^22 (half a turn of bias): the low 23 bits of tb are the
// phase mod one turn, offset so that [0, 2^23) maps to [-pi, pi); OR-ing them under the exponent of 2^23 makes
// the float 2^23 + (tb mod 2^23) without a conversion.
__device__ __forceinline__ void sincos_biased(int32_t tb, float* s, float* c) {
  const float f = __int_as_float((tb & 0x7FFFFF) | 0x4B000000);
  const float x = (f - 12582912.f) * (3.14159265358979323846f / PHI_ONE);      // 12582912 = 2^23 + 2^22
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(*s) : "f"(x));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(*c) : "f"(x));
}

// the same in three instructions before the SFU: one LOP3 ((tb & kmask) | kexp, the constants in registers) and one
// FMA (the rounded constant -3 pi shifts every pixel by the same 1e-7 rad, which no |.|^2 output sees)
__device__ __forceinline__ void sincos_biased_fma(int32_t tb, int32_t kmask, int32_t kexp, float* s, float* c) {
  int32_t u;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(u) : "r"(tb), "r"(kmask), "r"(kexp));
  constexpr float sc = 3.14159265358979323846f / PHI_ONE;
  const float x = fmaf(__int_as_float(u), sc, -12582912.f * sc);
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(*s) : "f"(x));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(*c) : "f"(x));
}

// sincos_biased_fma of two pixels, the FMA packed: (cos, sin) of each
__device__ __forceinline__ void sincos_biased_fma2(int32_t tb0, int32_t tb1, int32_t kmask, int32_t kexp, float2* cs0,
                                                   float2* cs1) {
  int32_t u0, u1;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(u0) : "r"(tb0), "r"(kmask), "r"(kexp));
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(u1) : "r"(tb1), "r"(kmask), "r"(kexp));
  constexpr float sc = 3.14159265358979323846f / PHI_ONE;
  const float2 x = f2_fma(make_float2(__int_as_float(u0), __int_as_float(u1)), make_float2(sc, sc),
                          make_float2(-12582912.f * sc, -12582912.f * sc));
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(cs0->y) : "f"(x.x));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cs0->x) : "f"(x.x));
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(cs1->y) : "f"(x.y));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cs1->x) : "f"(x.y));
}

__device__ __forceinline__ void split_pack2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 f = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - f.x, b - f.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

struct FieldParams {
  int num_envs;          // envs in this chunk
  int num_items;         // env blocks x Np NSEG column segments
  int items_per_cta;
  int nkb;               // KPAD / 64
  int col_origin;
  int env0;              // first env of the chunk (index into the tiles)
  int dbg;               // AOG_FK_DEBUG bits (tuning experiments only): 1 no phi stores, 2 no prefetch, 4 no TMEM load
  uint32_t sci_ratio_q32; // lambda_wfs / lambda_sci in 0.32 fixed point
  const uint16_t* apmask;
  const float2* m1o32;   // [n][Np] first obs-arm table, FP32
  float* phi;            // [env][Np / 16][Np x][16 y] total phase out, radians in [-pi, pi)
  float2* R4;            // [env][Np x][NSEG FK_PARTS][n] obs-arm column partial sums out (part s FK_PARTS + q)
  double2* strehl_part;  // [env][FK_SLOTS]
  const void* gfib;      // fused kernel: [Np x][Np / 16][16 y] per-pixel records (FK_NT float2 or FK_NF floats each)
  double2* fib_part;     // fused kernel: [env][FK_SLOTS][FK_JT] partial projection sums out
  int* err_flag;
};

// NP = pupil pixels per side: 240 (the reference, AO_env.py:216) for every mode; 128, 256 and 512 for the fused modes
// (BASELINE configs[4], the pupil-grid axis).  Any multiple of 16 up to 256 fits the tiles (N of the MMA, TMEM columns);
// 512 runs every column as two 256-pixel segments.
template <bool STREHL, int NOBS, int MODE, int NP = TC_NP>
// (448 threads x 144 registers would fit the register file on paper, but warps are allocated in groups of four: a
// build with __maxnreg__(144) fails to launch every variant above 128 registers.  The Strehl + 5x5-detector variant
// sits at that cap: it spilled 16 bytes (0.53 ms against 0.41 for either feature alone) until LATE_TILE below: 0.51.)
__global__ void __launch_bounds__(FK_THREADS, 1)
k_dm_phase_tc(const __grid_constant__ CUtensorMap tmAct_hi, const __grid_constant__ CUtensorMap tmAct_lo,
              const __grid_constant__ CUtensorMap tmM_hi, const __grid_constant__ CUtensorMap tmM_lo,
              const __grid_constant__ CUtensorMap tmHwt, const FieldParams p) {
  constexpr bool FUSED = MODE == 1 || MODE == 2, SYM = MODE == 2, PHASE_ONLY = MODE == 3;
  static_assert(NP % 16 == 0 && (NP <= 256 || (FUSED && NP == 512)), "pupil size of the phase kernel");
  constexpr int Np = NP;
  constexpr int NSEG = FK_NSEG(NP), SEG = NP / NSEG, IPB = NP * NSEG;   // segments per column, pixels each, items per env block
  constexpr uint32_t TX_BYTES = 2 * FK_A_TILE + 2 * SEG * 64 * 2;
  constexpr uint32_t IDESC = umma_idesc_f16(128, SEG);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // stays a shared-space pointer
  uint8_t* pf = base + FK_STAGES * FK_STAGE_BYTES;                       // phase prefetch rings, [FK_PARTS][FK_PF_STAGES]
  constexpr int PF_SLOT = FK_PF_SLOT(NOBS, MODE);
  constexpr int NT = FK_NT(NOBS);
  uint8_t* aux = pf + FK_PF_BYTES(NOBS, MODE);
  uint64_t* full = reinterpret_cast<uint64_t*>(aux);
  uint64_t* empty = full + FK_STAGES;
  uint64_t* tmem_full = empty + FK_STAGES;       // [2]
  uint64_t* tmem_empty = tmem_full + 2;          // [2]
  uint64_t* pf_full = tmem_empty + 2;            // [FK_PARTS][FK_PF_STAGES]
  uint64_t* pf_empty = pf_full + FK_PARTS * FK_PF_STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(pf_empty + FK_PARTS * FK_PF_STAGES);
  constexpr int NRED = FUSED ? 1 + FK_JT : 1;                            // Strehl sum + fibre projections
  double2* sred = reinterpret_cast<double2*>(aux + FK_AUX_BAR);          // [NRED][FK_PARTS][128 envs]
  float2* m1o_s = reinterpret_cast<float2*>(sred + NRED * FK_PARTS * 128);   // [n][Np] (not used by the fused kernel)
  // [Np][Np / 16] (read by the MODE 0 chunk loop only: not staged for the fused kernel)
  uint16_t* apmask_s = reinterpret_cast<uint16_t*>(m1o_s + (FUSED ? 0 : NOBS * Np));
  // [Np NSEG][2]: first lit chunk (index within the whole column), lit count of the segment
  uint8_t* run_s = reinterpret_cast<uint8_t*>(apmask_s + (FUSED ? 0 : Np * (Np / 16)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item_lo = blockIdx.x * p.items_per_cta;
  const int item_hi = min(p.num_items, item_lo + p.items_per_cta);

  if (!FUSED && !PHASE_ONLY)
    for (int i = threadIdx.x; i < NOBS * Np; i += blockDim.x) m1o_s[i] = p.m1o32[i];
  if (!FUSED)
    for (int i = threadIdx.x; i < Np * (Np / 16); i += blockDim.x) apmask_s[i] = p.apmask[i];
  for (int xs = threadIdx.x; xs < Np * NSEG; xs += blockDim.x) {
    const int c0 = (xs % NSEG) * (SEG / 16);
    int first = c0, cnt = 0;
    for (int c = c0; c < c0 + SEG / 16; ++c)
      if (p.apmask[(xs / NSEG) * (Np / 16) + c]) { if (!cnt) first = c; ++cnt; }
    run_s[2 * xs] = (uint8_t)first;
    run_s[2 * xs + 1] = (uint8_t)cnt;     // the aperture is convex: the lit chunks are contiguous
  }
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < FK_PARTS * FK_PF_STAGES; ++s) { mbar_init(&pf_full[s], 1); mbar_init(&pf_empty[s], 4); }
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmHwt)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmAct_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmAct_lo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmM_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmM_lo)) : "memory");
    for (int s = 0; s < FK_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], FK_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = item_lo; item < item_hi; ++item) {
        const int eb = item / IPB, xs = fk_segment<MODE, NP>(item - eb * IPB);
        const int row0 = (xs / NSEG) * Np + (xs % NSEG) * SEG;               // modes rows of pixels (x, s SEG ...)
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait<200>(&empty[stage], phase ^ 1, p.err_flag, 11);
          mbar_expect_tx(&full[stage], TX_BYTES);
          const uint32_t s0 = smem_u32(base + stage * FK_STAGE_BYTES);
          tma_load_2d(s0, &tmAct_hi, &full[stage], kb * 64, eb * 128);
          tma_load_2d(s0 + FK_A_TILE, &tmAct_lo, &full[stage], kb * 64, eb * 128);
          tma_load_2d(s0 + 2 * FK_A_TILE, &tmM_hi, &full[stage], kb * 64, row0);
          tma_load_2d(s0 + 2 * FK_A_TILE + FK_B_TILE, &tmM_lo, &full[stage], kb * 64, row0);
          if (++stage == FK_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int item = item_lo; item < item_hi; ++item, ++it) {
        const int as = it & 1;
        mbar_wait<200>(&tmem_empty[as], ((it >> 1) & 1) ^ 1, p.err_flag, 12);
        tc_fence_after();
        const uint32_t d = tmem_base + as * 256;
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait<100>(&full[stage], phase, p.err_flag, 13);
          tc_fence_after();
          const uint32_t s0 = smem_u32(base + stage * FK_STAGE_BYTES);
          // The tensor core truncates its FP32 accumulation (~ -0.5 ulp of the running sum per MMA): issue the
          // tiny hi.lo + lo.hi corrections FIRST, while the accumulator is still small, and the hi.hi chain last,
          // so only the 4 main MMAs of a K block round at the magnitude of the result.
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t a_hi = umma_desc_sw128(s0 + ks * 32);
            const uint64_t a_lo = umma_desc_sw128(s0 + FK_A_TILE + ks * 32);
            const uint64_t b_hi = umma_desc_sw128(s0 + 2 * FK_A_TILE + ks * 32);
            const uint64_t b_lo = umma_desc_sw128(s0 + 2 * FK_A_TILE + FK_B_TILE + ks * 32);
            tc_mma_f16(d, a_hi, b_lo, IDESC, (kb | ks) != 0);
            tc_mma_f16(d, a_lo, b_hi, IDESC, 1);
          }
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t a_hi = umma_desc_sw128(s0 + ks * 32);
            const uint64_t b_hi = umma_desc_sw128(s0 + 2 * FK_A_TILE + ks * 32);
            tc_mma_f16(d, a_hi, b_hi, IDESC, 1);
          }
          tc_commit(&empty[stage]);
          if (++stage == FK_STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit(&tmem_full[as]);
      }
    }
  } else {
    // ===================== epilogue: one env per thread =====================
    const int ew = warp - 2;                  // 0..11
    const int lg = warp & 3;                  // TMEM lane group this warp may touch
    const int q = ew >> 2;                    // takes lit chunks first + q, first + q + 3, ... of every column
    const int row = lg * 32 + lane;           // env within the block
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
    double st_re = 0.0, st_im = 0.0;
    int m_base = 0;                                    // lit chunks of the CTA's earlier items (mod FK_PARTS)
    double fb_re[FK_JT], fb_im[FK_JT];                 // fused kernel: fibre projection sums of my env
#pragma unroll
    for (int j = 0; j < FK_JT; ++j) fb_re[j] = fb_im[j] = 0.0;
    int cur_eb = -1;
    int it = 0;

    // The lit chunks of all of the CTA's items form ONE stream dealt round-robin to the FK_PARTS warps of a lane
    // group (chunk g of the stream -> warp g % FK_PARTS), so the warps stay within one chunk of each other over
    // the whole kernel instead of per item; the double-buffered accumulator absorbs the per-item difference.
    //
    // Phase prefetch: the four warps of a q group (one per lane group) walk the same sub-stream, so they share a
    // ring of FK_PF_STAGES slots.  Fill k of the group's sub-stream (its four 2 KB phase tiles, one tensor copy, and
    // its record tile) is issued by the group's warp with lg == k % 4, when that warp starts chunk k - 1; every warp
    // waits on full[k % S] before it reads chunk k and arrives once on empty[k % S] after it.
    // Progress: the issue of fill k waits on empty for chunk k - S <= k - 2, which every warp of the group reaches
    // before chunk k - 1; a warp waits on full[k] only after it has itself passed chunk k - 1, and so has issued
    // fill k if it is the issuer.  Take the group's lowest chunk m: its warps wait either on full[m] (issued, as the
    // issuer is at >= m), on empty for chunk m + 1 - S < m (read by all), on tmem_full (items before its own), or at
    // flush_strehl's bar.sync 1.  None of these waits on a warp that is parked at a later chunk or at bar.sync 1:
    // the bar.sync before item i needs only the chunks of items < i and the one fill issued ahead across it, whose
    // empty wait covers chunks of items < i.
    int n_item = item_lo - 1, n_ci = 0, n_end = 0;       // prefetch cursor: chunk n_ci of item n_item
    int n_x = 0, n_base = 0, n_cnt = 0;                  // its column, lit chunks before the item (mod FK_PARTS), its lit count
    auto next_lit = [&]() -> bool {
      n_ci += FK_PARTS;
      while (n_ci >= n_end) {
        n_base = (n_base + n_cnt) % FK_PARTS;
        if (++n_item >= item_hi) return false;
        const int n_xs = fk_segment<MODE, NP>(n_item - (n_item / IPB) * IPB);
        n_x = n_xs / NSEG;
        n_cnt = run_s[2 * n_xs + 1];
        n_ci = run_s[2 * n_xs] + (q + FK_PARTS - n_base) % FK_PARTS;
        n_end = run_s[2 * n_xs] + n_cnt;
      }
      return true;
    };
    uint8_t* const ring = pf + q * (FK_PF_STAGES * PF_SLOT);
    uint64_t* const rfull = pf_full + q * FK_PF_STAGES;
    uint64_t* const rempty = pf_empty + q * FK_PF_STAGES;
    int r_slot = 0, f_slot = 0, f_turn = 0;              // slot of the chunk being read; slot and issuer (k % 4) of fill k
    uint32_t r_phase = 0, f_phase = 0;
    // fill for the chunk at the cursor
    auto issue_fill = [&]() {
      if (f_turn == lg && lane == 0) {
        mbar_wait(&rempty[f_slot], f_phase ^ 1, p.err_flag, 16);
        int xp2 = n_x + p.col_origin;
        if (xp2 >= Np) xp2 -= Np;
        const int eb32 = (p.env0 + (n_item / IPB) * 128) >> 5;
        const uint32_t dst = smem_u32(ring + f_slot * PF_SLOT);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&rfull[f_slot], FK_PF_PHASE + FK_TAB_TILE(NOBS, MODE));
        asm volatile(
            "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %3, %4, %5, %6}], [%2];"
            ::"r"(dst), "l"(reinterpret_cast<uint64_t>(&tmHwt)), "r"(smem_u32(&rfull[f_slot])), "r"(0), "r"(n_ci), "r"(xp2),
              "r"(eb32) : "memory");
        if (FUSED) {
          const uint8_t* gsrc = static_cast<const uint8_t*>(p.gfib) + ((size_t)n_x * (Np / 16) + n_ci) * FK_TAB_TILE(NOBS, MODE);
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(dst + FK_PF_PHASE), "l"(gsrc), "r"((uint32_t)FK_TAB_TILE(NOBS, MODE)), "r"(smem_u32(&rfull[f_slot])) : "memory");
        }
      }
      f_turn = (f_turn + 1) & 3;
      if (++f_slot == FK_PF_STAGES) { f_slot = 0; f_phase ^= 1; }
    };
    bool n_ok = next_lit();
    if (n_ok && !(p.dbg & 2)) issue_fill();

    auto flush_strehl = [&](int eb) {
      // combine the thirds of every env, one partial per (env, CTA slot)
      if (STREHL) sred[q * 128 + row] = make_double2(st_re, st_im);
      if (FUSED) {
#pragma unroll
        for (int j = 0; j < FK_JT; ++j) sred[((1 + j) * FK_PARTS + q) * 128 + row] = make_double2(fb_re[j], fb_im[j]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(FK_EPI_WARPS * 32) : "memory");
      if (q == 0) {
        const int env = eb * 128 + row;
        if (env < p.num_envs) {
          const int slot = blockIdx.x - (eb * IPB) / p.items_per_cta;
          if (STREHL) {
            double2 a = sred[row];
            for (int k = 1; k < FK_PARTS; ++k) { a.x += sred[k * 128 + row].x; a.y += sred[k * 128 + row].y; }
            p.strehl_part[(size_t)env * FK_SLOTS + slot] = a;
          }
          if (FUSED) {
#pragma unroll
            for (int j = 0; j < FK_JT; ++j) {
              double2 a = sred[(1 + j) * FK_PARTS * 128 + row];
              for (int k = 1; k < FK_PARTS; ++k) {
                a.x += sred[((1 + j) * FK_PARTS + k) * 128 + row].x;
                a.y += sred[((1 + j) * FK_PARTS + k) * 128 + row].y;
              }
              p.fib_part[((size_t)env * FK_SLOTS + slot) * FK_JT + j] = a;
            }
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(FK_EPI_WARPS * 32) : "memory");
      st_re = st_im = 0.0;
#pragma unroll
      for (int j = 0; j < FK_JT; ++j) fb_re[j] = fb_im[j] = 0.0;
    };

    for (int item = item_lo; item < item_hi; ++item, ++it) {
      const int eb = item / IPB, xs = fk_segment<MODE, NP>(item - eb * IPB);
      const int x = xs / NSEG, seg = xs % NSEG;
      if ((STREHL || FUSED) && eb != cur_eb) {
        if (cur_eb >= 0) flush_strehl(cur_eb);
        cur_eb = eb;
      }
      const int as = it & 1;
      const int env = eb * 128 + row;
      mbar_wait(&tmem_full[as], (it >> 1) & 1, p.err_flag, 14);
      tc_fence_after();
      const bool valid = env < p.num_envs;
      // This item's sums over my chunks (at most 5 = 80 pixels) in FP32, folded into FP64 once per item: obs-arm
      // (re, im) per row, MODE 2: (ac, bs, as, bc) per conjugate pair, (ac, as) centre; fibre projections; Strehl.
      constexpr int NPP = SYM ? 4 * (NOBS / 2) + 2 * (NOBS & 1) : 2 * NOBS;
      float pp[NPP], fre[FK_JT], fim[FK_JT];
#pragma unroll
      for (int v = 0; v < NPP; ++v) pp[v] = 0.f;
#pragma unroll
      for (int k = 0; k < FK_JT; ++k) fre[k] = fim[k] = 0.f;
      constexpr int kmask = 0x7FFFFF, kexp = 0x4B000000;
      float sre = 0.f, sim = 0.f;
      const int run_first = run_s[2 * xs], run_end = run_first + run_s[2 * xs + 1];
      const int my_first = run_first + (q + FK_PARTS - m_base) % FK_PARTS;   // my chunks of the stream in this item
      m_base = (m_base + run_s[2 * xs + 1]) % FK_PARTS;
#pragma unroll 1
      for (int ci = my_first; ci < run_end; ci += FK_PARTS) {            // warp-uniform: only lit chunks
        const uint32_t mask = FUSED ? 0u : apmask_s[x * (Np / 16) + ci];
        const int y0 = ci * 16;
        float d[16];
        // pixel y of the column is accumulator column y - seg SEG of the segment's MMA
        if (!(p.dbg & 4)) tc_ld16(lane_addr + as * 256 + y0 - seg * SEG, d);
        else { for (int j = 0; j < 16; ++j) d[j] = 0.01f * j; }
        // this chunk's fill was issued one chunk ago; issue the next lit chunk's fill now if it is this warp's turn
        if (!(p.dbg & 2)) {
          n_ok = next_lit();
          if (n_ok) issue_fill();
          mbar_wait(&rfull[r_slot], r_phase, p.err_flag, 15);
        }
        const uint8_t* const slot_ptr = ring + r_slot * PF_SLOT;
        const uint8_t* tile = slot_ptr + lg * FK_PF_TILE + lane * 64;
        const int sw = (lane >> 1) & 3;                                   // pieces were stored at j ^ ((env >> 1) & 3)
        // The Strehl + wide-detector variants sit at the 128-register cap of a 448-thread block: they fetch the second
        // half of the phase tile after the first eight pixels instead of holding all 16 values through the loop.
        constexpr bool LATE_TILE = SYM && STREHL && NOBS >= 5;
        int32_t t[16];
#pragma unroll
        for (int j = 0; j < (LATE_TILE ? 2 : 4); ++j) {
          const int4 h = *reinterpret_cast<const int4*>(tile + ((j ^ sw) << 4));
          t[4 * j] = h.x; t[4 * j + 1] = h.y; t[4 * j + 2] = h.z; t[4 * j + 3] = h.w;
        }
        tc_wait_ld();
        if constexpr (SYM) {
          // ---- fused kernel, symmetric tables: 12 FMAs per pixel for the obs pair, the three fibre modes and Strehl.
          // The pixels go in pairs: the phase rounding and the angle FMA of the two are packed FP32x2 operations.
          constexpr int NP2 = NOBS / 2, NC = NOBS & 1, NF = FK_NF(NOBS);
          const float4* tab = reinterpret_cast<const float4*>(slot_ptr + FK_PF_PHASE);   // [16 y][NF / 4]
          const int32_t q31 = (int32_t)(p.sci_ratio_q32 >> 1);
          const int32_t sci_bias = (1 << 22) - 2 * (int32_t)(((long long)(1 << 22) * (long long)q31) >> 32);
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            if (LATE_TILE && j == 8) {
#pragma unroll
              for (int jj = 2; jj < 4; ++jj) {
                const int4 h = *reinterpret_cast<const int4*>(tile + ((jj ^ sw) << 4));
                t[4 * jj] = h.x; t[4 * jj + 1] = h.y; t[4 * jj + 2] = h.z; t[4 * jj + 3] = h.w;
              }
            }
            int32_t tb[2];
            phase_fixed_rn2(d[j], d[j + 1], &tb[0], &tb[1]);
            tb[0] += t[j] + (1 << 22);
            tb[1] += t[j + 1] + (1 << 22);
            float2 e[2], es[2];                                             // (cos, sin) at lambda_wfs, lambda_sci
            sincos_biased_fma2(tb[0], tb[1], kmask, kexp, &e[0], &e[1]);
            if (STREHL)
              sincos_biased_fma2(2 * __mulhi(tb[0], q31) + sci_bias, 2 * __mulhi(tb[1], q31) + sci_bias, kmask, kexp,
                                 &es[0], &es[1]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const float c0 = e[h].x, s0 = e[h].y;
              float4 rec[NF / 4];
#pragma unroll
              for (int r = 0; r < NF / 4; ++r) rec[r] = tab[(j + h) * (NF / 4) + r];
              const float* m = reinterpret_cast<const float*>(rec);
#pragma unroll
              for (int v = 0; v < NP2; ++v) {
                pp[4 * v + 0] = fmaf(m[2 * v], c0, pp[4 * v + 0]);
                pp[4 * v + 1] = fmaf(m[2 * v + 1], s0, pp[4 * v + 1]);
                pp[4 * v + 2] = fmaf(m[2 * v], s0, pp[4 * v + 2]);
                pp[4 * v + 3] = fmaf(m[2 * v + 1], c0, pp[4 * v + 3]);
              }
              if (NC) {
                pp[4 * NP2] = fmaf(m[2 * NP2], c0, pp[4 * NP2]);
                pp[4 * NP2 + 1] = fmaf(m[2 * NP2], s0, pp[4 * NP2 + 1]);
              }
#pragma unroll
              for (int k = 0; k < FK_JT; ++k) {
                fre[k] = fmaf(m[2 * NP2 + NC + k], c0, fre[k]);
                fim[k] = fmaf(m[2 * NP2 + NC + k], s0, fim[k]);
              }
              if (STREHL) {
                sre = fmaf(m[2 * NP2 + NC + FK_JT], es[h].x, sre);
                sim = fmaf(m[2 * NP2 + NC + FK_JT], es[h].y, sim);
              }
            }
          }
        } else if constexpr (FUSED) {
          // ---- fused kernel: the whole optics chain of these 16 pixels, nothing leaves the SM
          const float4* tab = reinterpret_cast<const float4*>(slot_ptr + FK_PF_PHASE);   // [16 y][NT / 2]
          const int32_t q31 = (int32_t)(p.sci_ratio_q32 >> 1);
          // 2 mulhi(tb, q31) + sci_bias = (t lambda_wfs / lambda_sci) + 2^22, with tb = t + 2^22
          const int32_t sci_bias = (1 << 22) - 2 * (int32_t)(((long long)(1 << 22) * (long long)q31) >> 32);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            // atmosphere + DM in fixed point (2^22 per half-turn, unreduced), biased by half a turn
            const int32_t tb = t[j] + phase_fixed_rn(d[j]) + (1 << 22);
            float c0, s0;
            sincos_biased(tb, &s0, &c0);
            float4 rec[NT / 2];
#pragma unroll
            for (int r = 0; r < NT / 2; ++r) rec[r] = tab[j * (NT / 2) + r];
            const float2* m = reinterpret_cast<const float2*>(rec);   // [obs rows | fibre modes | (aperture, 0)]
#pragma unroll
            for (int v = 0; v < NOBS; ++v) {
              pp[2 * v] = fmaf(m[v].x, c0, fmaf(-m[v].y, s0, pp[2 * v]));
              pp[2 * v + 1] = fmaf(m[v].x, s0, fmaf(m[v].y, c0, pp[2 * v + 1]));
            }
            // c_j = sum_pixels E . G_j (AO_env.py:471 through the back-projected mode)
#pragma unroll
            for (int k = 0; k < FK_JT; ++k) {
              fre[k] = fmaf(m[NOBS + k].x, c0, fmaf(-m[NOBS + k].y, s0, fre[k]));
              fim[k] = fmaf(m[NOBS + k].x, s0, fmaf(m[NOBS + k].y, c0, fim[k]));
            }
            if (STREHL) {
              // phase at lambda_sci = phase at lambda_wfs x (lambda_wfs / lambda_sci), to two fixed-point units
              const int32_t ts = 2 * __mulhi(tb, q31) + sci_bias;
              float cs, ss;
#ifdef AOG_FK_NO_STREHL_MUFU       // tuning build: how much of the kernel is the SFU pipe
              cs = __int_as_float((ts & 0x7FFFFF) | 0x3F000000); ss = cs;
#else
              sincos_biased(ts, &ss, &cs);
#endif
              sre = fmaf(m[NOBS + FK_JT].x, cs, sre);
              sim = fmaf(m[NOBS + FK_JT].x, ss, sim);
            }
          }
        } else {
          float ph[16];                                                     // total phase at lambda_wfs, [-pi, pi)
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            t[j] += phase_fixed_rn(d[j]);                                   // atmosphere + DM, fixed point, unreduced
            ph[j] = small_int_to_float((t[j] << 9) >> 9) * (3.14159265358979323846f / PHI_ONE);
          }
          if (!(p.dbg & 1)) {
            // Full-sector stores: a lane's 16 pixels are 64 contiguous bytes, but a thread stores at most 16 per
            // instruction.  Lane pairs swap halves so that each store instruction writes whole 32-byte sectors
            // (lanes 2i, 2i+1 -> the two halves of a sector of env 2i, then of env 2i+1).
            const bool odd = lane & 1;
            const bool valid_even = (env & ~1) < p.num_envs, valid_odd = (env | 1) < p.num_envs;
            float* row_even = p.phi + (((size_t)(env & ~1) * (Np / 16) + ci) * Np + x) * 16 + (odd ? 4 : 0);
            float* row_odd = row_even + (size_t)Np * Np;
#pragma unroll
            for (int h8 = 0; h8 < 2; ++h8) {              // pixels [8 h8, 8 h8 + 8) = one sector per env
              const float* a = ph + 8 * h8;
              float r[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) r[k] = __shfl_xor_sync(0xffffffffu, odd ? a[k] : a[4 + k], 1);
              // even lane: own[0..3] -> env 2i first half;  received = env 2i+1's first half
              // odd lane : received = env 2i's second half;  own[4..7] -> env 2i+1 second half
              if (valid_even)
                *reinterpret_cast<float4*>(row_even + 8 * h8) = odd ? make_float4(r[0], r[1], r[2], r[3]) : make_float4(a[0], a[1], a[2], a[3]);
              if (valid_odd)
                *reinterpret_cast<float4*>(row_odd + 8 * h8) = odd ? make_float4(a[4], a[5], a[6], a[7]) : make_float4(r[0], r[1], r[2], r[3]);
            }
          }
          if constexpr (!PHASE_ONLY) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float c0, s0;
              asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s0) : "f"(ph[j]));
              asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c0) : "f"(ph[j]));
              if (mask != 0xFFFFu && !((mask >> j) & 1u)) { c0 = 0.f; s0 = 0.f; }
#pragma unroll
              for (int v = 0; v < NOBS; ++v) {
                const float2 m = m1o_s[v * Np + y0 + j];
                pp[2 * v] = fmaf(m.x, c0, fmaf(-m.y, s0, pp[2 * v]));
                pp[2 * v + 1] = fmaf(m.x, s0, fmaf(m.y, c0, pp[2 * v + 1]));
              }
            }
          }
          if (STREHL) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              // phase at lambda_sci = phase at lambda_wfs x (lambda_wfs / lambda_sci), exact to one fixed-point unit
              const int32_t ts = (int32_t)(((long long)t[j] * (long long)p.sci_ratio_q32) >> 32);
              float c0, s0;
              sincos_fixed(ts, &s0, &c0);
              if (mask == 0xFFFFu || ((mask >> j) & 1u)) { sre += c0; sim += s0; }
            }
          }
        }
        if (!(p.dbg & 2)) {
          __syncwarp();                                                   // every lane has read the slot
          if (lane == 0) mbar_arrive(&rempty[r_slot]);
        }
        if (++r_slot == FK_PF_STAGES) { r_slot = 0; r_phase ^= 1; }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);       // this warp is done with the accumulator
      if (valid && !PHASE_ONLY) {
        float2* r = p.R4 + (((size_t)env * Np + x) * (NSEG * FK_PARTS) + seg * FK_PARTS + q) * NOBS;
        if constexpr (SYM) {
          // pair v: row v = (ac - bs, as + bc), row n-1-v = (ac + bs, as - bc)
          constexpr int NP2 = NOBS / 2;
#pragma unroll
          for (int v = 0; v < NP2; ++v) {
            const double ac = pp[4 * v], bs = pp[4 * v + 1], as_ = pp[4 * v + 2], bc = pp[4 * v + 3];
            r[v] = make_float2((float)(ac - bs), (float)(as_ + bc));
            r[NOBS - 1 - v] = make_float2((float)(ac + bs), (float)(as_ - bc));
          }
          if (NOBS & 1) r[NP2] = make_float2(pp[4 * NP2], pp[4 * NP2 + 1]);
        } else {
#pragma unroll
          for (int v = 0; v < NOBS; ++v) r[v] = make_float2(pp[2 * v], pp[2 * v + 1]);
        }
      }
      if (FUSED) {
#pragma unroll
        for (int k = 0; k < FK_JT; ++k) { fb_re[k] += (double)fre[k]; fb_im[k] += (double)fim[k]; }
      }
      if (STREHL) { st_re += (double)sre; st_im += (double)sim; }
    }
    if ((STREHL || FUSED) && cur_eb >= 0) flush_strehl(cur_eb);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ----------------------------------------------------------------------------- fused optics, tiny batches
// k_small_fused: the fused optics chain (k_dm_phase_tc MODE 2: same tables, same fixed-point phase, same sums) for
// batches of at most SMALL_MAX envs -- BASELINE configs[0] is literally ONE env.  The tensor-core kernel gives a
// 128-env block to every pupil column and one env to every thread, so for a single env 127 of 128 lanes idle through
// 240 x 15 chunks (26 us); here a THREAD IS A PIXEL: a CTA takes `ipc` pupil columns, thread y forms the DM phase of
// pixel (x, y) for every env as an FP32 dot product over the split-fp16 operands the tensor cores would read (a_hi +
// a_lo and m_hi + m_lo are exact in FP32), adds the atmosphere tile, takes sin / cos on the SFU and multiplies with
// its record; the column sums are reduced in FP64 (warp shuffles, then the 8 warps through shared memory).  Outputs
// have the layout k_finalize_tcw reads: R4[env][x][part 0] (parts 1, 2 zero) and one Strehl / fibre slot per CTA.
constexpr int SMALL_MAX = 8;
struct SmallParams {
  int B, Np, kpad, ipc, col_origin, env0;
  uint32_t sci_ratio_q32;
  const int32_t* hwt; const uint16_t* apmask; const float* gfib;
  const __half* act_hi; const __half* act_lo; const __half* m_hi; const __half* m_lo;
  float2* R4; double2* strehl_part; double2* fib_part;
};
template <bool STREHL, int NOBS>
__global__ void __launch_bounds__(256) k_small_fused(const SmallParams p) {
  constexpr int NP2 = NOBS / 2, NC = NOBS & 1, NF = FK_NF(NOBS);
  constexpr int NO = 4 * NP2 + 2 * NC, NV = NO + 2 * FK_JT + 2;      // obs products | fibre (re, im) | Strehl (re, im)
  __shared__ float act_s[SMALL_MAX][128];
  __shared__ double red_s[8][SMALL_MAX][NV];
  __shared__ double fin_s[SMALL_MAX][NV];
  __shared__ double slot_s[SMALL_MAX][2 * FK_JT + 2];
  const int Np = p.Np, y = threadIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < SMALL_MAX * 128; i += 256) {
    const int b = i >> 7, k = i & 127;
    act_s[b][k] = (b < p.B && k < p.kpad)
                      ? __half2float(p.act_hi[(size_t)b * p.kpad + k]) + __half2float(p.act_lo[(size_t)b * p.kpad + k]) : 0.f;
  }
  for (int i = threadIdx.x; i < SMALL_MAX * (2 * FK_JT + 2); i += 256) (&slot_s[0][0])[i] = 0.0;
  __syncthreads();
  constexpr int kmask = 0x7FFFFF, kexp = 0x4B000000;
  const int32_t q31 = (int32_t)(p.sci_ratio_q32 >> 1);
  const int32_t sci_bias = (1 << 22) - 2 * (int32_t)(((long long)(1 << 22) * (long long)q31) >> 32);
  for (int xi = 0; xi < p.ipc; ++xi) {
    const int x = blockIdx.x * p.ipc + xi;
    if (x >= Np) break;
    const bool lit = y < Np && ((p.apmask[x * (Np / 16) + (y >> 4)] >> (y & 15)) & 1);
    float d[SMALL_MAX];
#pragma unroll
    for (int b = 0; b < SMALL_MAX; ++b) d[b] = 0.f;
    float rec[NF];
    if (lit) {
      const size_t pix = (size_t)x * Np + y;
      for (int kb = 0; kb < p.kpad; kb += 64) {
        float m[64];
        const uint4* mh = reinterpret_cast<const uint4*>(p.m_hi + pix * p.kpad + kb);
        const uint4* ml = reinterpret_cast<const uint4*>(p.m_lo + pix * p.kpad + kb);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 h = __ldg(mh + c), l = __ldg(ml + c);
          const __half2* hh = reinterpret_cast<const __half2*>(&h);
          const __half2* ll = reinterpret_cast<const __half2*>(&l);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 fh = __half22float2(hh[e]), fl = __half22float2(ll[e]);
            m[8 * c + 2 * e] = fh.x + fl.x;
            m[8 * c + 2 * e + 1] = fh.y + fl.y;
          }
        }
#pragma unroll
        for (int b = 0; b < SMALL_MAX; ++b) {
          if (b < p.B) {
            float acc = d[b];
#pragma unroll
            for (int k4 = 0; k4 < 16; ++k4) {
              const float4 a = *reinterpret_cast<const float4*>(&act_s[b][kb + 4 * k4]);
              acc = fmaf(a.x, m[4 * k4], acc); acc = fmaf(a.y, m[4 * k4 + 1], acc);
              acc = fmaf(a.z, m[4 * k4 + 2], acc); acc = fmaf(a.w, m[4 * k4 + 3], acc);
            }
            d[b] = acc;
          }
        }
      }
      const float4* rp = reinterpret_cast<const float4*>(p.gfib + pix * NF);
#pragma unroll
      for (int r = 0; r < NF / 4; ++r) {
        const float4 v = __ldg(rp + r);
        rec[4 * r] = v.x; rec[4 * r + 1] = v.y; rec[4 * r + 2] = v.z; rec[4 * r + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int r = 0; r < NF; ++r) rec[r] = 0.f;
    }
    int xp = x + p.col_origin;
    if (xp >= Np) xp -= Np;
#pragma unroll
    for (int b = 0; b < SMALL_MAX; ++b) {
      if (b >= p.B) break;                                          // uniform
      double vals[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) vals[v] = 0.0;
      if (lit) {
        const int env = p.env0 + b, l = env & 31;
        const size_t ti = (((size_t)(env >> 5) * Np + xp) * (Np / 16) + (y >> 4)) * 512 + (size_t)l * 16 +
                          ((((y >> 2) & 3) ^ ((l >> 1) & 3)) << 2) + (y & 3);
        const int32_t tb = __ldg(p.hwt + ti) + __float2int_rn(d[b] * PHI_ONE) + (1 << 22);
        float c0, s0;
        sincos_biased_fma(tb, kmask, kexp, &s0, &c0);
#pragma unroll
        for (int v = 0; v < NP2; ++v) {
          vals[4 * v + 0] = (double)(rec[2 * v] * c0);
          vals[4 * v + 1] = (double)(rec[2 * v + 1] * s0);
          vals[4 * v + 2] = (double)(rec[2 * v] * s0);
          vals[4 * v + 3] = (double)(rec[2 * v + 1] * c0);
        }
        if (NC) { vals[4 * NP2] = (double)(rec[2 * NP2] * c0); vals[4 * NP2 + 1] = (double)(rec[2 * NP2] * s0); }
#pragma unroll
        for (int k = 0; k < FK_JT; ++k) {
          vals[NO + 2 * k] = (double)(rec[2 * NP2 + NC + k] * c0);
          vals[NO + 2 * k + 1] = (double)(rec[2 * NP2 + NC + k] * s0);
        }
        if (STREHL) {
          const int32_t ts = 2 * __mulhi(tb, q31) + sci_bias;
          float cs, ss;
          sincos_biased_fma(ts, kmask, kexp, &ss, &cs);
          vals[NO + 2 * FK_JT] = (double)(rec[2 * NP2 + NC + FK_JT] * cs);
          vals[NO + 2 * FK_JT + 1] = (double)(rec[2 * NP2 + NC + FK_JT] * ss);
        }
      }
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const double sum = warp_sum(vals[v]);
        if (lane == 0) red_s[warp][b][v] = sum;
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < p.B * NV; i += 256) {
      const int b = i / NV, v = i - b * NV;
      double sum = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) sum += red_s[w][b][v];
      fin_s[b][v] = sum;
      if (v >= NO) slot_s[b][v - NO] += sum;                       // the same thread owns (b, v) for every column
    }
    __syncthreads();
    // column sums of the obs arm: pair v -> rows v and n-1-v, as k_dm_phase_tc MODE 2 forms them
    for (int i = threadIdx.x; i < p.B * NOBS * FK_PARTS; i += 256) {
      const int b = i / (NOBS * FK_PARTS), r = i - b * (NOBS * FK_PARTS), q = r / NOBS, v = r - q * NOBS;
      float2 out = make_float2(0.f, 0.f);
      if (q == 0) {
        const double* f = fin_s[b];
        if (NC && v == NP2) out = make_float2((float)f[4 * NP2], (float)f[4 * NP2 + 1]);
        else if (v < NP2) out = make_float2((float)(f[4 * v] - f[4 * v + 1]), (float)(f[4 * v + 2] + f[4 * v + 3]));
        else { const int w = NOBS - 1 - v; out = make_float2((float)(f[4 * w] + f[4 * w + 1]), (float)(f[4 * w + 2] - f[4 * w + 3])); }
      }
      p.R4[(((size_t)b * Np + x) * FK_PARTS + q) * NOBS + v] = out;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.B * (FK_JT + 1); i += 256) {
    const int b = i / (FK_JT + 1), j = i - b * (FK_JT + 1);
    const double2 v = make_double2(slot_s[b][2 * j], slot_s[b][2 * j + 1]);
    if (j < FK_JT) p.fib_part[((size_t)b * FK_SLOTS + blockIdx.x) * FK_JT + j] = v;
    else if (STREHL) p.strehl_part[(size_t)b * FK_SLOTS + blockIdx.x] = v;
  }
}

// ----------------------------------------------------------------------------- field + MFT stage 1
// k_field_mft1: the pupil field is formed ON CHIP and fed straight into the stage-1 pair MMA
// (reference AO_env.py:132-135 field, :138 first MFT product):
//
//   [Tr ; Ti] (256 x 240) = [[M1r, -M1i], [M1i, M1r]] (256 x 480) . [Er ; Ei] (480 x 240)      per env
//
// cta_group::2, M = 256 over the CTA pair (CTA 0: Tr rows, CTA 1: Ti rows), N = 240 pupil columns x, CTA r
// stages x in [120 r, 120 r + 120).  The K order is 15 blocks of [16 y real | 16 y imaginary].  16 warps:
//   warp 0      TMA producer of the twiddle tiles (A): a deep ring (8 x 16 KB) because every tile is an
//               L2 round trip; completion on the leader's `a_full` barrier
//   warp 1      MMA issuer (leader CTA only)
//   warps 4-11  epilogue: TMEM -> registers -> accumulators released -> split fp16 -> smem ring -> TMA store
//   warp 2      TMA producer of the phase tiles (120 columns x 16 y, FP32 radians, SWIZZLE_64B ring of 6): the
//               field warps must not have global loads of their own in flight, because the release fence of
//               their barrier arrival waits for them
//   warps 12-15 field warps, one pupil column x per thread: phase -> sincos (SFU) -> aperture -> fp16 hi/lo
//               split -> the B operand rows, written in the UMMA SWIZZLE_64B image.  They work on PAIRS of
//               K blocks (one B slot = 2 x 16 KB, ring of 2) so the fence + barrier traffic is paid once
//               per 32 pixels; `b_full` collects one arrival per field warp of BOTH CTAs
// Registers are re-partitioned with setmaxnreg: the epilogue warps hold 128 accumulator columns each.
#ifndef AOG_F1_A_SLOTS        // ring depths: overridable for tuning builds (make EXTRA=-DAOG_F1_A_SLOTS=...)
#define AOG_F1_A_SLOTS 4
#endif
#ifndef AOG_F1_B_SLOTS
#define AOG_F1_B_SLOTS 2
#endif
#ifndef AOG_F1_PHI_SLOTS
#define AOG_F1_PHI_SLOTS 6
#endif
constexpr int F1_A_SLOTS = AOG_F1_A_SLOTS;
constexpr int F1_B_SLOTS = AOG_F1_B_SLOTS;            // each holds a PAIR of K blocks
constexpr int F1_SLOT_BYTES = 2 * A_TILE;             // 16 KB: [hi 8 KB][lo 8 KB] of one K block
constexpr int F1_PHI_SLOTS = AOG_F1_PHI_SLOTS;
constexpr int F1_PHI_TILE = 8192;                     // 120 rows x 64 B in an 8 KB slot
constexpr int F1_THREADS = 512;
constexpr int F1_SMEM_BYTES = (F1_A_SLOTS + 2 * F1_B_SLOTS) * F1_SLOT_BYTES + F1_PHI_SLOTS * F1_PHI_TILE + M2_EPI_BYTES +
                              1024 /*align*/ + 1024 /*barriers*/;

struct F1Params {
  int num_items;            // envs in this chunk
  const uint16_t* apmask;   // [Np x][Np / 16] aperture bits
  int dbg;                  // AOG_TC_DEBUG bits: 1 no MMA, 4 no epilogue work, 32 no field arithmetic, 64 no phase tiles, 128 no twiddle tiles
  int* err_flag;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F1_THREADS, 1)
k_field_mft1(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
             const __grid_constant__ CUtensorMap tmPhi, const __grid_constant__ CUtensorMap tmO_hi,
             const __grid_constant__ CUtensorMap tmO_lo, const F1Params p) {
  constexpr int B_ROWS = TC_NP / 2;                                    // 120 rows of B per CTA
  constexpr uint32_t TX_BYTES = 2 * 2 * A_TILE;                        // A tiles of both CTAs
  constexpr uint32_t IDESC = umma_idesc_f16(256, TC_NP);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_ring = base;
  uint8_t* b_ring = base + F1_A_SLOTS * F1_SLOT_BYTES;
  uint8_t* phis = b_ring + 2 * F1_B_SLOTS * F1_SLOT_BYTES;             // phase tile ring
  uint8_t* epi = phis + F1_PHI_SLOTS * F1_PHI_TILE;                    // output tile ring
  uint64_t* a_full = reinterpret_cast<uint64_t*>(epi + M2_EPI_BYTES);
  uint64_t* a_empty = a_full + F1_A_SLOTS;
  uint64_t* b_full = a_empty + F1_A_SLOTS;
  uint64_t* b_empty = b_full + F1_B_SLOTS;
  uint64_t* phi_full = b_empty + F1_B_SLOTS;
  uint64_t* phi_empty = phi_full + F1_PHI_SLOTS;
  uint64_t* tmem_full = phi_empty + F1_PHI_SLOTS;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_lo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmPhi)) : "memory");
    for (int s = 0; s < F1_A_SLOTS; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < F1_B_SLOTS; ++s) { mbar_init(&b_full[s], 8); mbar_init(&b_empty[s], 1); }
    for (int s = 0; s < F1_PHI_SLOTS; ++s) { mbar_init(&phi_full[s], 1); mbar_init(&phi_empty[s], 4); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 2 * M2_EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0 && lane == 0) {
      // ===================== TMA producer: twiddle tiles =====================
      int slot = 0;
      uint32_t phase = 0;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait<32>(&a_empty[slot], phase ^ 1, p.err_flag, 1);
          if (p.dbg & 128) {
            if (rank == 0) mbar_arrive(&a_full[slot]);
          } else {
            if (rank == 0) mbar_expect_tx(&a_full[slot], TX_BYTES);
            const uint32_t s0 = smem_u32(a_ring + slot * F1_SLOT_BYTES);
            const uint32_t fb = mapa_rank(smem_u32(&a_full[slot]), 0);
            tma_load_2d_pair(s0, &tmA_hi, fb, kb * KB, (int)rank * 128);
            tma_load_2d_pair(s0 + A_TILE, &tmA_lo, fb, kb * KB, (int)rank * 128);
          }
          if (++slot == F1_A_SLOTS) { slot = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1 && rank == 0 && lane == 0) {
      // ===================== MMA issuer (one thread of the leader CTA) =====================
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0, tphase = 0;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        mbar_wait<32>(tmem_empty, tphase ^ 1, p.err_flag, 2);
        tc_fence_after();
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait(&a_full[sa], pa, p.err_flag, 3);
          if (!(kb & 1)) mbar_wait(&b_full[sb], pb, p.err_flag, 8);       // a B slot carries K blocks kb, kb + 1
          tc_fence_after();
          const uint32_t a0 = smem_u32(a_ring + sa * F1_SLOT_BYTES);
          const uint32_t b0 = smem_u32(b_ring + (2 * sb + (kb & 1)) * F1_SLOT_BYTES);
          if (!(p.dbg & 1))
#pragma unroll
          for (int ks = 0; ks < KB / 16; ++ks) {
            const uint32_t acc = (kb | ks) != 0;
            const uint64_t a_hi = umma_desc_sw64(a0 + ks * 32), a_lo = umma_desc_sw64(a0 + A_TILE + ks * 32);
            const uint64_t b_hi = umma_desc_sw64(b0 + ks * 32), b_lo = umma_desc_sw64(b0 + A_TILE + ks * 32);
            tc_mma_f16_pair(tmem_base, a_hi, b_hi, IDESC, acc);              // main
            tc_mma_f16_pair(tmem_base + 256, a_hi, b_lo, IDESC, acc);        // corrections
            tc_mma_f16_pair(tmem_base + 256, a_lo, b_hi, IDESC, 1);
          }
          tc_commit_pair(&a_empty[sa]);             // the slot is free in both CTAs when these MMAs retire
          if (++sa == F1_A_SLOTS) { sa = 0; pa ^= 1; }
          if ((kb & 1) || kb == NUM_KB - 1) {
            tc_commit_pair(&b_empty[sb]);
            if (++sb == F1_B_SLOTS) { sb = 0; pb ^= 1; }
          }
        }
        tc_commit_pair(tmem_full);
        tphase ^= 1;
      }
    } else if (warp == 2 && lane == 0 && !(p.dbg & 64)) {
      // ===================== TMA producer: phase tiles of my 120 pupil columns =====================
      int slot = 0;
      uint32_t phase = 0;
      for (int item = cluster_id; item < p.num_items; item += num_clusters) {
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait<32>(&phi_empty[slot], phase ^ 1, p.err_flag, 5);
          mbar_expect_tx(&phi_full[slot], B_ROWS * 64);
          tma_load_2d(smem_u32(phis + slot * F1_PHI_TILE), &tmPhi, &phi_full[slot], 0,
                      (item * NUM_KB + kb) * TC_NP + (int)rank * B_ROWS);
          if (++slot == F1_PHI_SLOTS) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp < 12) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    // ===================== epilogue: 8 warps, TMEM lane group = warp % 4, column half = (warp - 4) / 4 =========
    const int lg = warp & 3;
    const int half = (warp - 4) >> 2;
    const int row = lg * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
    const uint32_t tmem_empty_leader = mapa_rank(smem_u32(tmem_empty), 0);
    uint32_t tphase = 0;
    uint32_t out_seq = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters) {
      mbar_wait(tmem_full, tphase, p.err_flag, 4);
      tc_fence_after();
      tphase ^= 1;
      if (p.dbg & 4) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tmem_empty_leader);
        continue;
      }
      // Phase 1: drain this warp's accumulator columns (main + corrections) into registers and hand the
      // TMEM back, so the next env's MMAs run under phase 2.  The 4 warps of a column half own the
      // 16-column chunks c = 8 half ... (8 | 7 of the 15).
      const int c0 = half * 8, c_end = half ? TC_NP / 16 : 8;
      float acc[128];
#pragma unroll
      for (int i = 0; i < 8; i += 2) {
        float v[32], w[32];
        if (c0 + i + 1 < c_end) {
          tc_ld32(lane_addr + (c0 + i) * 16, v);
          tc_ld32(lane_addr + 256 + (c0 + i) * 16, w);
        } else {
          tc_ld16(lane_addr + (c0 + i) * 16, v);
          tc_ld16(lane_addr + 256 + (c0 + i) * 16, w);
#pragma unroll
          for (int q = 16; q < 32; ++q) v[q] = w[q] = 0.f;
        }
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 32; ++q) acc[i * 16 + q] = v[q] + w[q];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty_leader);
      // Phase 2: split fp16 -> swizzled 128 x 16 tiles in shared memory -> TMA stores into
      // T[env][v][k = rank * 240 + x].
      uint8_t* ring = epi + half * (M2_OUT_BUFS * 2 * M2_OUT_TILE);
      const uint32_t sw = (uint32_t)((row >> 2) & 1);                 // SWIZZLE_32B: 16-byte piece ^= address bit 7
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = c0 + i;
        if (c < c_end) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) split_pack2(acc[i * 16 + 2 * q], acc[i * 16 + 2 * q + 1], hi[q], lo[q]);
          uint8_t* t_hi = ring + (out_seq % M2_OUT_BUFS) * (2 * M2_OUT_TILE);
          uint8_t* t_lo = t_hi + M2_OUT_TILE;
          *reinterpret_cast<uint4*>(t_hi + row * 32 + ((0u ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(t_hi + row * 32 + ((1u ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          *reinterpret_cast<uint4*>(t_lo + row * 32 + ((0u ^ sw) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(t_lo + row * 32 + ((1u ^ sw) << 4)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          if (half == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
          else           asm volatile("bar.sync 2, 128;" ::: "memory");
          if (lg == 0 && lane == 0) {
            tma_store_2d(&tmO_hi, smem_u32(t_hi), (int)rank * TC_NP + c * 16, item * 128);
            tma_store_2d(&tmO_lo, smem_u32(t_lo), (int)rank * TC_NP + c * 16, item * 128);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            // the store issued one chunk ago has left shared memory: with 3 buffers the slot written two
            // chunks from now is free by the time its writers pass the next barrier
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          }
          ++out_seq;
        }
      }
    }
    if (lg == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores landed
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 128;");
    // ===================== field warps: one pupil column x per thread =====================
    const int t = (warp - 12) * 32 + lane;                 // B row within this CTA's half
    const bool active = t < B_ROWS;
    const int x = active ? (int)rank * B_ROWS + t : (int)rank * B_ROWS;
    const uint32_t sw = (uint32_t)((t >> 1) & 3);          // SWIZZLE_64B: 16-byte piece ^= (row >> 1) & 3
    const uint32_t b_full_leader0 = mapa_rank(smem_u32(&b_full[0]), 0);
    uint32_t maskw[8];                                     // aperture bits of my column, two 16-pixel chunks per word
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t lo16 = __ldg(p.apmask + x * (TC_NP / 16) + 2 * j);
      const uint32_t hi16 = (2 * j + 1 < TC_NP / 16) ? __ldg(p.apmask + x * (TC_NP / 16) + 2 * j + 1) : 0u;
      maskw[j] = lo16 | (hi16 << 16);
    }
    int sb = 0, slot = 0;
    uint32_t pb = 0, pphase = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters) {
#pragma unroll
      for (int kb = 0; kb < NUM_KB; ++kb) {                  // fully unrolled: kb indexes the mask registers
        if (!(p.dbg & 64)) mbar_wait(&phi_full[slot], pphase, p.err_flag, 6);
        if (!(kb & 1)) mbar_wait(&b_empty[sb], pb ^ 1, p.err_flag, 7);
        if (active && !(p.dbg & 32)) {
          const uint32_t mask = (kb & 1) ? (maskw[kb >> 1] >> 16) : (maskw[kb >> 1] & 0xFFFFu);
          uint8_t* b_hi = b_ring + (2 * sb + (kb & 1)) * F1_SLOT_BYTES + t * 64;
          uint8_t* b_lo = b_hi + A_TILE;
          if (mask == 0) {                                  // outside the aperture: the field is zero
            const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              *reinterpret_cast<uint4*>(b_hi + (j << 4)) = z;
              *reinterpret_cast<uint4*>(b_lo + (j << 4)) = z;
            }
          } else {
            const uint8_t* tile = phis + slot * F1_PHI_TILE + t * 64;
#pragma unroll
            for (int h8 = 0; h8 < 2; ++h8) {                // pixels [8 h8, 8 h8 + 8) of the chunk
              const float4 q0 = *reinterpret_cast<const float4*>(tile + (((uint32_t)(2 * h8) ^ sw) << 4));
              const float4 q1 = *reinterpret_cast<const float4*>(tile + (((uint32_t)(2 * h8 + 1) ^ sw) << 4));
              const float ph[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
              float c[8], s[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s[j]) : "f"(ph[j]));
                asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c[j]) : "f"(ph[j]));
              }
              if (mask != 0xFFFFu) {                        // aperture edge: clear the dark pixels
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  if (!((mask >> (8 * h8 + j)) & 1u)) { c[j] = 0.f; s[j] = 0.f; }
              }
              uint32_t rh[4], rl[4], ih[4], il[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                split_pack2(c[2 * j], c[2 * j + 1], rh[j], rl[j]);
                split_pack2(s[2 * j], s[2 * j + 1], ih[j], il[j]);
              }
              // row image: [16 y real | 16 y imaginary] = pieces {0, 1 | 2, 3}; this half fills piece h8 of each
              *reinterpret_cast<uint4*>(b_hi + (((uint32_t)h8 ^ sw) << 4)) = make_uint4(rh[0], rh[1], rh[2], rh[3]);
              *reinterpret_cast<uint4*>(b_hi + (((uint32_t)(2 + h8) ^ sw) << 4)) = make_uint4(ih[0], ih[1], ih[2], ih[3]);
              *reinterpret_cast<uint4*>(b_lo + (((uint32_t)h8 ^ sw) << 4)) = make_uint4(rl[0], rl[1], rl[2], rl[3]);
              *reinterpret_cast<uint4*>(b_lo + (((uint32_t)(2 + h8) ^ sw) << 4)) = make_uint4(il[0], il[1], il[2], il[3]);
            }
          }
        }
        if ((kb & 1) || kb == NUM_KB - 1) {                   // the pair is complete: publish it
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            mbar_arrive_cluster(b_full_leader0 + sb * 8);     // my rows of the B tiles are in place
            if (!(p.dbg & 64)) {                              // the phase tiles may be overwritten
              if (kb & 1) mbar_arrive(&phi_empty[slot == 0 ? F1_PHI_SLOTS - 1 : slot - 1]);
              mbar_arrive(&phi_empty[slot]);
            }
          }
          if (++sb == F1_B_SLOTS) { sb = 0; pb ^= 1; }
        }
        if (++slot == F1_PHI_SLOTS) { slot = 0; pphase ^= 1; }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  // neither CTA may exit (or free its TMEM) while the pair's MMAs, loads or barrier signals can still touch it
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// Action -> actuators (AO_env.py:115-120) with the GEMM A operand written in the same pass: one warp per env, the
// Gram matrix of the modes (var(M a) = a^T G a, np.std over the whole grid) staged once per block in shared memory
// and read transposed (G is symmetric) so that lanes hit consecutive banks.  a_hi / a_lo rows >= B and columns
// >= K stay zero from allocation.
template <typename ActT>
__global__ void __launch_bounds__(256)
k_actuators_pack(const ActT* __restrict__ actions, const double* __restrict__ gram, double* __restrict__ act,
                 __half* __restrict__ a_hi, __half* __restrict__ a_lo, int B, int K, int kpad, int sh_operation,
                 double target_rms, double pack_scale) {
  extern __shared__ double sh_g[];                     // [K][K] Gram + [8 warps][K] actions
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* A = sh_g + (size_t)K * K + warp * K;
  if (!sh_operation)
    for (int i = threadIdx.x; i < K * K; i += blockDim.x) sh_g[i] = gram[i];
  __syncthreads();
  for (int b = blockIdx.x * 8 + warp; b < B; b += gridDim.x * 8) {
    for (int k = lane; k < K; k += 32) {
      const double a = (double)actions[(size_t)b * K + k];
      A[k] = sh_operation ? a : a / (double)(k + 10);
    }
    __syncwarp();
    double scale = 1.0;
    if (!sh_operation) {
      double part = 0.0;
      for (int i = lane; i < K; i += 32) {
        // four independent chains: the 64-term dot product was one dependent FP64 FMA chain per lane (latency bound)
        double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
        int j = 0;
        for (; j + 3 < K; j += 4) {
          r0 = fma(sh_g[(size_t)j * K + i], A[j], r0);
          r1 = fma(sh_g[(size_t)(j + 1) * K + i], A[j + 1], r1);
          r2 = fma(sh_g[(size_t)(j + 2) * K + i], A[j + 2], r2);
          r3 = fma(sh_g[(size_t)(j + 3) * K + i], A[j + 3], r3);
        }
        for (; j < K; ++j) r0 = fma(sh_g[(size_t)j * K + i], A[j], r0);
        part += A[i] * ((r0 + r1) + (r2 + r3));
      }
      scale = target_rms / sqrt(fmax(warp_sum(part), 0.0));   // var == 0 -> inf -> 0 * inf = NaN (reference semantics); never sqrt(-eps)
    }
    for (int k = lane; k < K; k += 32) {
      const double v = A[k] * scale;
      act[(size_t)b * K + k] = v;
      const double w = v * pack_scale;
      const __half h = __float2half_rn((float)w);
      a_hi[(size_t)b * kpad + k] = h;
      a_lo[(size_t)b * kpad + k] = __float2half_rn((float)(w - (double)__half2float(h)));
    }
    __syncwarp();
  }
}

// actuators (FP64, after normalisation) -> GEMM A operand: half-turn scale, split fp16, zero padded
__global__ void k_act_pack(const double* __restrict__ act, __half* __restrict__ a_hi, __half* __restrict__ a_lo,
                           int K, int kpad, int env0, int nB, int rows, double scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * kpad) return;
  const int r = i / kpad, k = i - r * kpad;
  const double v = (r < nB && k < K) ? act[(size_t)(env0 + r) * K + k] * scale : 0.0;
  const __half h = __float2half_rn((float)v);
  a_hi[i] = h;
  a_lo[i] = __float2half_rn((float)(v - (double)__half2float(h)));
}

// screens FP64 [B][xp][y] -> tiled fixed-point phase at lambda_wfs (layout: TensorState::hwt).
// One thread per output int, output-ordered (coalesced writes, strided reads).  factor != null (aog_set_turbulence's
// rescale): each env's screen is first multiplied in place by factor[env], and the tile is that of the product, so it
// equals what a later plain conversion of the rescaled screens would write.
__device__ __forceinline__ int32_t phase_fixed(double S, double inv) {
  double a = S * inv * (double)PHI_ONE;                  // half-turns x 2^22
  a = fmin(fmax(a, -2147483000.0), 2147483000.0);        // +-512 half-turns (1600 rad) of range
  return (int32_t)__double2ll_rn(a);
}
__global__ void k_screens_to_tiles(double* __restrict__ src, int32_t* __restrict__ hwt, int Np, int B,
                                   size_t total, double inv_w, const double* __restrict__ factor) {
  const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= total) return;
  const int e = o & 3, piece = (o >> 2) & 3, l = (o >> 4) & 31;
  const size_t t = o >> 9;                        // ((eb32 * Np) + xp) * (Np / 16) + ci
  const int ci = (int)(t % (Np / 16));
  const size_t t2 = t / (Np / 16);
  const int xp = (int)(t2 % Np);
  const size_t env = (t2 / Np) * 32 + l;
  const int y = ci * 16 + ((piece ^ ((l >> 1) & 3)) << 2) + e;
  int32_t v = 0;
  if (env < (size_t)B) {
    double* s = src + (env * Np + xp) * Np + y;                                      // screens are [env][x][y]
    double S = *s;
    if (factor) *s = S = S * factor[env];
    v = phase_fixed(S, inv_w);
  }
  hwt[o] = v;
}

// k_finalize_tcw<N, PARTS>: the epilogue of the tensor / fused paths, R4 holding PARTS partial column sums per
// contraction index, with ONE WARP per env and no block-level barrier.  The kernel is bound by the LATENCY of fetching
// the env's column partial sums (28.8 KB for the 5x5 detector), not by its arithmetic (DESIGN 4.6), so the partial
// sums stream through shared memory: every warp keeps a
// double-buffered ring of tiles (8 XS pupil columns = ~6 KB each, 16-byte cp.async, one commit group per tile) in
// flight ahead of its arithmetic -- 16 warps per SM x 6-12 KB outstanding.
// Lane (xs, b) = (lane / N, lane % N) owns column b of the column sums and the pupil columns x = xs, xs + XS, ...
// (XS = 32 / N): per x it adds the PARTS partial sums of R[x][b] in FP64 and multiplies them with the N table
// entries m[a][x] (broadcast loads), i.e. N complex accumulators per lane instead of N^2 -- no lane computes anything
// twice.  The XS partial results per detector pixel meet in shared memory, summed in a fixed order by the lane that owns
// the pixel.  Slot sums (fibre projections, Strehl) are loaded before the contraction and reduced after it.
// Summation order depends on the env's data only: a batched env equals its single-env twin bit for bit.
constexpr int FIN_WARPS = 8;
template <int N, int PARTS> struct FinCfg {
  static constexpr int XS = 32 / N, LANES = XS * N, N2 = N * N, N2P = N2 < 7 ? 7 : N2;
  static constexpr int ITER = N >= 6 ? 4 : 8, TILE_X = XS * ITER, ROW = PARTS * N /* float2 per pupil column */;
  static constexpr int TAB_MAX = N * 512 * 16;           // the [N][Np] table, Np <= 512 on the tensor / fused paths
  static constexpr int TILE_BYTES = TILE_X * ROW * 8, WARP_BYTES = 2 * TILE_BYTES, SMEM = FIN_WARPS * WARP_BYTES;
  static constexpr int RED_LD = 33;
  static_assert(TILE_BYTES % 16 == 0, "tile size");
  static_assert((2 * N * RED_LD + 2 * N2P) * 8 <= WARP_BYTES, "the reduction scratch aliases the tile ring");
};
template <int N, int PARTS>
__global__ void __launch_bounds__(FIN_WARPS * 32, 2) k_finalize_tcw(FinalizeArgs a, int num_envs) {
  using Cfg = FinCfg<N, PARTS>;
  constexpr int XS = Cfg::XS, LANES = Cfg::LANES, N2 = Cfg::N2, ITER = Cfg::ITER, TILE_X = Cfg::TILE_X, ROW = Cfg::ROW;
  extern __shared__ __align__(16) unsigned char fin_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * FIN_WARPS + warp;
  unsigned char* wbase = fin_smem + warp * Cfg::WARP_BYTES;
  double2* tab_s = reinterpret_cast<double2*>(fin_smem + FIN_WARPS * Cfg::WARP_BYTES);   // [N][Np] second obs-arm table
  constexpr unsigned FULL = 0xffffffffu;
  const int ntiles = (a.Np + TILE_X - 1) / TILE_X;
  const float2* r4 = a.R4 + (size_t)b * a.Np * ROW;
  auto issue = [&](int t, int buf) {
    const int cols = min(TILE_X, a.Np - t * TILE_X);
    const int nchunks = cols * ROW / 2;                                // 16-byte pieces (cols is even)
    const unsigned char* src = reinterpret_cast<const unsigned char*>(r4 + (size_t)t * TILE_X * ROW);
    const unsigned dst = (unsigned)__cvta_generic_to_shared(wbase + buf * Cfg::TILE_BYTES);
    for (int c = lane; c < nchunks; c += 32)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + c * 16), "l"(src + (size_t)c * 16) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (b < num_envs) {
    issue(0, 0);
    if (ntiles > 1) issue(1, 1);
  }
  // the table is read N times per (pupil column, lane): from global memory those loads were the kernel's stall
  // (L1 hit rate 39 % next to 184 KB of shared memory; ncu: long scoreboard 6 of 14 warp-cycles per issue)
  for (int i = threadIdx.x; i < N * a.Np; i += FIN_WARPS * 32) tab_s[i] = __ldg(a.m1o + i);
  __syncthreads();
  if (b >= num_envs) return;                            // warps are independent from here on
  if (a.act) {
    int bad = 0;
    for (int k = lane; k < a.K; k += 32) bad |= isfinite(a.act[(size_t)b * a.K + k]) ? 0 : 1;   // inf: exp(i inf) = NaN too
    if (__any_sync(FULL, bad)) {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      const double qnan = __longlong_as_double(0x7ff8000000000000LL);
      for (int t = lane; t < N2; t += 32) {
        if (a.obs64) a.obs64[(size_t)b * N2 + t] = qnan;
        if (a.obs16) a.obs16[(size_t)b * N2 + t] = 0x7e00;
      }
      if (lane == 0 && a.compute_reward) {
        if (a.reward) a.reward[b] = qnan;
        if (a.power) a.power[b] = qnan;
        if (a.strehl) a.strehl[b] = qnan;
        if (a.ssim) a.ssim[b] = qnan;
      }
      return;
    }
  }
  // per-lane partial slot sums (reduced after the contraction)
  double2 cj[AOG_MAX_LP];
  double2 sp = make_double2(0.0, 0.0);
#pragma unroll
  for (int j = 0; j < AOG_MAX_LP; ++j) cj[j] = make_double2(0.0, 0.0);
  if (a.compute_reward) {
    const int eb = b >> 7;
    const int nslots = ((eb + 1) * a.slot_items - 1) / a.slot_ipc - (eb * a.slot_items) / a.slot_ipc + 1;
    if (a.coef_is_raw == 2) {
      if (lane == 0) {
#pragma unroll
        for (int j = 0; j < AOG_MAX_LP; ++j)
          if (j < a.J) {
            const double* c4 = a.coef4 + ((size_t)b * a.J + j) * 4;
            cj[j] = make_double2(c4[0] + c4[1], c4[2] + c4[3]);
          }
      }
    } else {
      const double2* fp = a.fib_part + (size_t)b * a.fib_slots * a.fib_stride;
      for (int i = lane; i < nslots; i += 32) {
#pragma unroll
        for (int j = 0; j < AOG_MAX_LP; ++j)
          if (j < a.J) { const double2 v = fp[i * a.fib_stride + j]; cj[j].x += v.x; cj[j].y += v.y; }
      }
    }
    if (a.rew_type == AOG_REW_STREHL_RATIO) {
      const double2* spp = a.strehl_part + (size_t)b * a.strehl_blocks;
      for (int i = lane; i < nslots; i += 32) { const double2 v = spp[i]; sp.x += v.x; sp.y += v.y; }
    }
  }
  // contraction over the pupil columns
  const int xs = lane / N, bb = lane - xs * N;
  double are[N], aim[N];
#pragma unroll
  for (int v = 0; v < N; ++v) are[v] = aim[v] = 0.0;
  for (int t = 0; t < ntiles; ++t) {
    if (t + 1 < ntiles) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else                asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    const float2* tile = reinterpret_cast<const float2*>(wbase + (t & 1) * Cfg::TILE_BYTES);
    if (lane < LANES) {
#pragma unroll
      for (int i = 0; i < ITER; ++i) {
        const int xl = xs + XS * i, x = t * TILE_X + xl;
        if (x < a.Np) {
          double ex = 0.0, ey = 0.0;
#pragma unroll
          for (int qq = 0; qq < PARTS; ++qq) {
            const float2 t4 = tile[(xl * PARTS + qq) * N + bb];
            ex += (double)t4.x;
            ey += (double)t4.y;
          }
#pragma unroll
          for (int v = 0; v < N; ++v) {
            const double2 m = tab_s[v * a.Np + x];
            are[v] = fma(m.x, ex, fma(-m.y, ey, are[v]));
            aim[v] = fma(m.x, ey, fma(m.y, ex, aim[v]));
          }
        }
      }
    }
    __syncwarp();
    if (t + 2 < ntiles) issue(t + 2, t & 1);
  }
  double* red = reinterpret_cast<double*>(wbase);               // [2 N][RED_LD]; the tile ring is drained
  double* obs_s = red + 2 * N * Cfg::RED_LD;
  double* win_s = obs_s + Cfg::N2P;
#pragma unroll
  for (int v = 0; v < N; ++v) { red[(2 * v) * Cfg::RED_LD + lane] = are[v]; red[(2 * v + 1) * Cfg::RED_LD + lane] = aim[v]; }
  __syncwarp();
  for (int t = lane; t < N2; t += 32) {
    const int v = t / N, u = t - v * N;
    double re = 0.0, im = 0.0;
#pragma unroll
    for (int s = 0; s < XS; ++s) { re += red[(2 * v) * Cfg::RED_LD + s * N + u]; im += red[(2 * v + 1) * Cfg::RED_LD + s * N + u]; }
    const double fr = re * a.norm.x - im * a.norm.y, fi = re * a.norm.y + im * a.norm.x;
    const double pw = (fr * fr + fi * fi) * a.obs_weight;
    const int to = u * N + v;          // R4 and the table (M2o^T) hold the transposed contraction
    obs_s[to] = pw;
    if (a.obs64) a.obs64[(size_t)b * N2 + to] = pw;
    if (a.obs16) a.obs16[(size_t)b * N2 + to] = __half_as_ushort(__double2half(pw));
  }
  __syncwarp();
  if (!a.compute_reward) return;
  // fibre: out = M (c e^{i beta L});  total power = c'^H G c'
  double2 c[AOG_MAX_LP];
#pragma unroll
  for (int j = 0; j < AOG_MAX_LP; ++j) {
    if (j < a.J) {
      double2 s = make_double2(warp_sum(cj[j].x), warp_sum(cj[j].y));
      s = make_double2(s.x * a.coef_scale.x - s.y * a.coef_scale.y, s.x * a.coef_scale.y + s.y * a.coef_scale.x);
      const double2 ph = a.lpphase[j];
      c[j] = make_double2(s.x * ph.x - s.y * ph.y, s.x * ph.y + s.y * ph.x);
    } else {
      c[j] = make_double2(0.0, 0.0);
    }
  }
  double power = 0.0;
#pragma unroll
  for (int j = 0; j < AOG_MAX_LP; ++j)
#pragma unroll
    for (int k = 0; k < AOG_MAX_LP; ++k)
      if (j < a.J && k < a.J) power += a.lpgram[j * a.J + k] * (c[j].x * c[k].x + c[j].y * c[k].y);
  double reward;
  if (a.rew_type == AOG_REW_STREHL_RATIO) {
    const double sr = warp_sum(sp.x), si = warp_sum(sp.y);
    const double strehl = a.strehl_scale * (sr * sr + si * si);
    if (lane == 0 && a.strehl) a.strehl[b] = strehl;
    reward = -(100.0 - strehl);
  } else {
    // skimage SSIM on 1-D data (ssim_1d, finalize.cuh), one window per lane, summed in window order
    const double peak = a.ssim_peak, C1 = (0.01 * peak) * (0.01 * peak), C2 = (0.03 * peak) * (0.03 * peak);
    const double cov_norm = 7.0 / 6.0;
    constexpr int ref_idx = N2 / 2;
    for (int cw = 3 + lane; cw < N2 - 3; cw += 32) {
      double sx = 0, sxx = 0, sy = 0, syy = 0, sxy = 0;
      for (int i = cw - 3; i <= cw + 3; ++i) {
        const double x = obs_s[i], r = (i == ref_idx) ? peak : 0.0;
        sx += x; sxx += x * x; sy += r; syy += r * r; sxy += x * r;
      }
      const double ux = sx / 7, uy = sy / 7, uxx = sxx / 7, uyy = syy / 7, uxy = sxy / 7;
      const double vx = cov_norm * (uxx - ux * ux), vy = cov_norm * (uyy - uy * uy), vxy = cov_norm * (uxy - ux * uy);
      win_s[cw] = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
    }
    __syncwarp();
    double tot = 0.0;
    for (int cw = 3; cw < N2 - 3; ++cw) tot += win_s[cw];      // same summation order as ssim_1d
    const double sv = tot / (double)(N2 - 6);
    if (lane == 0 && a.ssim) a.ssim[b] = sv;
    reward = 0.8 * power + (1.0 - 0.8) * sv;
  }
  if (lane != 0) return;
  if (a.has_thr && reward < a.thr) reward = -1.0;
  if (a.reward) a.reward[b] = reward;
  if (a.power) a.power[b] = power;
}

// ----------------------------------------------------------------------------- host helpers
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp16 row-major [rows][inner] tensor, box = box_inner x box_rows; box_inner * 2 B is the swizzle span
// (32 halves -> SWIZZLE_64B for the MFT operands, 64 halves -> SWIZZLE_128B for the DM GEMM operands).
int make_map(aog_env* env, CUtensorMap* map, const __half* ptr, uint64_t rows, uint32_t box_rows,
             uint64_t inner = TC_K, uint32_t box_inner = KB) {
  EncodeTiledFn enc = get_encode();
  if (!enc) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)inner * sizeof(__half)};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)ptr, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box_inner == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                   : (box_inner == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return AOG_OK;
}

// 2-D row-major [rows][inner] tensor of 32-bit words, box = 16 x box_rows (64-byte rows, SWIZZLE_64B)
int make_map_32(aog_env* env, CUtensorMap* map, const void* ptr, uint64_t rows, uint32_t box_rows, uint64_t inner) {
  EncodeTiledFn enc = get_encode();
  if (!enc) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)inner * sizeof(int32_t)};
  cuuint32_t box[2] = {16, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, (void*)ptr, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled (int32) failed: " + std::to_string((int)r));
  return AOG_OK;
}

// the phase tiles [blocks of 32 envs][Np][Np / 16][32][16] int32 (TensorState::hwt) as a 5-D tensor; box = the four
// 32-env tiles of one (column, chunk), 4 x 2 KB, copied as they are (the tiles are swizzled in memory already)
int make_map_hwt(aog_env* env, CUtensorMap* map, const int32_t* ptr, uint64_t blocks32, int Np) {
  EncodeTiledFn enc = get_encode();
  if (!enc) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  const uint64_t tile = 32 * 16 * sizeof(int32_t);
  cuuint64_t dims[5] = {16, 32, (cuuint64_t)Np / 16, (cuuint64_t)Np, (cuuint64_t)blocks32};
  cuuint64_t strides[4] = {16 * sizeof(int32_t), tile, tile * (Np / 16), tile * (Np / 16) * Np};
  cuuint32_t box[5] = {16, 32, 1, 1, 4};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_INT32, 5, (void*)ptr, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) AOG_FAIL(AOG_ERR_CUDA, "cuTensorMapEncodeTiled (phase tiles) failed: " + std::to_string((int)r));
  return AOG_OK;
}

void split_half(double x, __half* hi, __half* lo) {
  const __half h = __float2half_rn((float)x);
  *hi = h;
  *lo = __float2half_rn((float)(x - (double)__half2float(h)));
}

int upload_split(aog_env* env, const std::vector<double>& m, __half* d_hi, __half* d_lo) {
  std::vector<__half> hi(m.size()), lo(m.size());
  for (size_t i = 0; i < m.size(); ++i) split_half(m[i], &hi[i], &lo[i]);
  AOG_CUDA(cudaMemcpy(d_hi, hi.data(), hi.size() * sizeof(__half), cudaMemcpyHostToDevice));
  AOG_CUDA(cudaMemcpy(d_lo, lo.data(), lo.size() * sizeof(__half), cudaMemcpyHostToDevice));
  return AOG_OK;
}

}  // namespace

// =============================================================================================
int aog_tensor_create(aog_env* env) {
  const aog_config& c = env->cfg;
  const int NPc = c.num_pupil_pixels;
  if (c.precision == AOG_PRECISION_TENSOR && (NPc != TC_NP || c.num_focal_pixels != TC_NF))
    AOG_FAIL(AOG_ERR_UNSUPPORTED, "precision='tensor' (matrix-Fourier-transform GEMMs) is built for num_pupil_pixels=240, "
                                  "num_focal_pixels=128; use precision='fused' (pupil 128 / 240 / 256 / 512, any focal grid) "
                                  "or 'f64'");
  if (c.precision == AOG_PRECISION_FUSED && NPc != TC_NP &&
      !((NPc == 128 || NPc == 256 || NPc == 512) && (c.obs_dim == 2 || c.obs_dim == 5)))
    AOG_FAIL(AOG_ERR_UNSUPPORTED, "precision='fused' supports num_pupil_pixels=240 (any obs_dim <= 8) and 128 / 256 / 512 "
                                  "(obs_dim 2 or 5), with any focal grid; use precision='f64' for other grids");
  env->tensor.reset(new TensorState());
  TensorState* ts = env->tensor.get();
  ts->fused = c.precision == AOG_PRECISION_FUSED;
  if (ts->fused && c.num_lp_modes > FK_JT)
    AOG_FAIL(AOG_ERR_UNSUPPORTED, "fused precision path holds at most 3 guided fibre modes; use precision='tensor'");
  cudaDeviceProp prop;
  AOG_CUDA(cudaGetDeviceProperties(&prop, c.device));
  ts->num_sms = prop.multiProcessorCount;
  const size_t ch = env->chunk, B = c.num_envs, P = env->P;
  int rc;
#define A(expr) if ((rc = (expr))) return rc
  if (!ts->fused) {
    A(ts->A1_hi.alloc(env, (size_t)256 * TC_K));
    A(ts->A1_lo.alloc(env, (size_t)256 * TC_K));
    A(ts->B2_hi.alloc(env, (size_t)256 * TC_K));
    A(ts->B2_lo.alloc(env, (size_t)256 * TC_K));
    A(ts->phi.alloc(env, ch * P));
    AOG_CUDA(cudaMemset(ts->phi, 0, ch * P * sizeof(float)));   // out-of-aperture chunks are never written (nor used)
    // stage-2 reads env pairs: keep one spare env of rows so the last odd pair stays in bounds
    A(ts->T_hi.alloc(env, (ch + 1) * 128 * TC_K));
    A(ts->T_lo.alloc(env, (ch + 1) * 128 * TC_K));
    AOG_CUDA(cudaMemset(ts->T_hi, 0, (ch + 1) * 128 * TC_K * sizeof(__half)));
    AOG_CUDA(cudaMemset(ts->T_lo, 0, (ch + 1) * 128 * TC_K * sizeof(__half)));
    A(ts->lpw.alloc(env, (size_t)c.num_lp_modes * env->NF2));
    A(ts->lpwr.alloc(env, (size_t)c.num_lp_modes * env->NF2));
    A(ts->coef4.alloc(env, ch * (size_t)c.num_lp_modes * 4));
  } else {
    A(ts->gfib.alloc(env, (size_t)P * FK_NT(c.obs_dim)));
    AOG_CUDA(cudaMemset(ts->gfib, 0, (size_t)P * FK_NT(c.obs_dim) * sizeof(float2)));
    A(ts->fib_part.alloc(env, ch * (size_t)FK_SLOTS * FK_JT));
    A(ts->lpphase_f.alloc(env, (size_t)AOG_MAX_LP));
  }
  if (c.obs_dim > 8) AOG_FAIL(AOG_ERR_UNSUPPORTED, "tensor precision path supports obs_dim <= 8");
  ts->kpad = ((c.num_modes + 63) / 64) * 64;
  ts->act_rows = (int)((ch + 127) / 128) * 128;
  {
    const size_t tiles = ((B + 127) / 128) * 4 * NPc * (NPc / 16);       // whole 128-env blocks: the prefetch reads them all
    A(ts->hwt.alloc(env, tiles * 512));
    AOG_CUDA(cudaMemset(ts->hwt, 0, tiles * 512 * sizeof(int32_t)));
    A(make_map_hwt(env, &ts->tmHwt, ts->hwt, tiles / ((size_t)NPc * (NPc / 16)), NPc));
    env->phase_tiles = ts->hwt;
    env->phase_tiles_unit = (double)PHI_ONE;
  }
  A(ts->modesK_hi.alloc(env, P * ts->kpad));
  A(ts->modesK_lo.alloc(env, P * ts->kpad));
  A(ts->act_hi.alloc(env, (size_t)ts->act_rows * ts->kpad));
  A(ts->act_lo.alloc(env, (size_t)ts->act_rows * ts->kpad));
  AOG_CUDA(cudaMemset(ts->act_hi, 0, (size_t)ts->act_rows * ts->kpad * sizeof(__half)));
  AOG_CUDA(cudaMemset(ts->act_lo, 0, (size_t)ts->act_rows * ts->kpad * sizeof(__half)));
  A(ts->apmask.alloc(env, (size_t)NPc * (NPc / 16)));
  A(ts->m1o32.alloc(env, (size_t)c.obs_dim * NPc));
  A(ts->R4.alloc(env, ch * NPc * FK_NSEG(NPc) * FK_PARTS * c.obs_dim));
  A(ts->m2oT.alloc(env, (size_t)c.obs_dim * NPc));
  // barrier-timeout code: mapped pinned HOST memory, so that the host can still read it after the trap that follows
  // a timeout has poisoned the CUDA context (aog_health)
  AOG_CUDA(ts->err_flag_host.alloc(1, cudaHostAllocMapped));
  *ts->err_flag_host = 0;
  AOG_CUDA(cudaHostGetDevicePointer((void**)&ts->err_flag, ts->err_flag_host, 0));
  if (!ts->fused) {
    A(make_map(env, &ts->tmA1_hi, ts->A1_hi, 256, 128));
    A(make_map(env, &ts->tmA1_lo, ts->A1_lo, 256, 128));
    A(make_map_32(env, &ts->tmPhi, ts->phi, ch * (TC_NP / 16) * TC_NP, TC_NP / 2, 16));   // box = 120 columns x 16 y, contiguous
    A(make_map(env, &ts->tmT128_hi, ts->T_hi, (ch + 1) * 128, 128));
    A(make_map(env, &ts->tmT128_lo, ts->T_lo, (ch + 1) * 128, 128));
    A(make_map(env, &ts->tmTout_hi, ts->T_hi, (ch + 1) * 128, 128, TC_K, 16));
    A(make_map(env, &ts->tmTout_lo, ts->T_lo, (ch + 1) * 128, 128, TC_K, 16));
    A(make_map(env, &ts->tmB2_hi, ts->B2_hi, 256, 128));
    A(make_map(env, &ts->tmB2_lo, ts->B2_lo, 256, 128));
  }
  A(make_map(env, &ts->tmAct_hi, ts->act_hi, ts->act_rows, 128, ts->kpad, 64));
  A(make_map(env, &ts->tmAct_lo, ts->act_lo, ts->act_rows, 128, ts->kpad, 64));
  // B operand of the phase kernel: one column segment of pixels (a TMA box holds at most 256 rows)
  A(make_map(env, &ts->tmModes_hi, ts->modesK_hi, P, NPc / FK_NSEG(NPc), ts->kpad, 64));
  A(make_map(env, &ts->tmModes_lo, ts->modesK_lo, P, NPc / FK_NSEG(NPc), ts->kpad, 64));
#undef A
  AOG_CUDA(cudaFuncSetAttribute(k_mft2<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, M2_SMEM_BYTES));
  AOG_CUDA(cudaFuncSetAttribute(k_mft2<AOG_MAX_LP>, cudaFuncAttributeMaxDynamicSharedMemorySize, M2_SMEM_BYTES));
  return AOG_OK;
}

namespace {
// Fibre modes propagated back to the pupil plane (FP64 on the host):
//   c_j = norm sum_{v,u} (mode_j w)[v][u] F[v][u],   F = M1 . E . M2   (AO_env.py:138, :471)
//       = norm sum_{y,x} E[y][x] G_j[y][x],          G_j = M1^T (mode_j w) M2^T
// so the coupling coefficients are J inner products over the pupil and the focal plane is never formed.
int build_backprojected_modes(aog_env* env, TensorState* ts) {
  const int Np = env->cfg.num_pupil_pixels, Nf = env->cfg.num_focal_pixels, J = env->cfg.num_lp_modes;
  const std::vector<double>&m1 = ts->h_m1, &m2 = ts->h_m2, &lp = ts->h_lp;
  std::vector<double> H((size_t)2 * Nf * Np), G((size_t)2 * J * Np * Np);
  double gmax = 0.0;
  for (int j = 0; j < J; ++j) {
    for (int v = 0; v < Nf; ++v)                       // H[v][x] = sum_u lp[j][v][u] M2[x][u]
      for (int x = 0; x < Np; ++x) {
        double re = 0.0, im = 0.0;
        const double* w = &lp[((size_t)j * Nf + v) * Nf];
        const double* b = &m2[(size_t)2 * x * Nf];
        for (int u = 0; u < Nf; ++u) { re += w[u] * b[2 * u]; im += w[u] * b[2 * u + 1]; }
        H[2 * ((size_t)v * Np + x)] = re;
        H[2 * ((size_t)v * Np + x) + 1] = im;
      }
    for (int y = 0; y < Np; ++y)                       // G[y][x] = sum_v M1[v][y] H[v][x]
      for (int x = 0; x < Np; ++x) {
        double re = 0.0, im = 0.0;
        for (int v = 0; v < Nf; ++v) {
          const double ar = m1[2 * ((size_t)v * Np + y)], ai = m1[2 * ((size_t)v * Np + y) + 1];
          const double hr = H[2 * ((size_t)v * Np + x)], hi = H[2 * ((size_t)v * Np + x) + 1];
          re += ar * hr - ai * hi;
          im += ar * hi + ai * hr;
        }
        G[2 * (((size_t)j * Np + y) * Np + x)] = re;
        G[2 * (((size_t)j * Np + y) * Np + x) + 1] = im;
        gmax = std::max(gmax, std::max(std::fabs(re), std::fabs(im)));
      }
  }
  if (gmax == 0.0) gmax = 1.0;
  ts->gfib_scale = gmax;
  // is every G_j one unit phasor times a real function?  (true on hcipy's symmetric grids)
  ts->g_real = true;
  for (int j = 0; j < J; ++j) {
    const double* g = &G[(size_t)2 * j * Np * Np];
    size_t imax = 0;
    double amax = 0.0;
    for (size_t i = 0; i < (size_t)Np * Np; ++i) {
      const double a = g[2 * i] * g[2 * i] + g[2 * i + 1] * g[2 * i + 1];
      if (a > amax) { amax = a; imax = i; }
    }
    const double th = std::atan2(g[2 * imax + 1], g[2 * imax]);
    ts->theta[j] = th;
    const double cr = std::cos(th), sr = std::sin(th);
    double res = 0.0;
    for (size_t i = 0; i < (size_t)Np * Np; ++i) res = std::max(res, std::fabs(g[2 * i + 1] * cr - g[2 * i] * sr));
    if (res > 1e-10 * std::sqrt(amax)) ts->g_real = false;
  }
  ts->h_G.swap(G);
  ts->have_G = true;
  return AOG_OK;
}

// per-pixel records of the fused kernel (TensorState::gfib), once G, the obs-arm table and the aperture are known
int build_fused_records(aog_env* env, TensorState* ts) {
  if (!(ts->have_G && ts->have_m1o && ts->have_ap && ts->have_lpphase)) return AOG_OK;
  const int Np = env->cfg.num_pupil_pixels, J = env->cfg.num_lp_modes, n = env->cfg.obs_dim, NT = FK_NT(n);
  // do the obs-arm rows come in conjugate pairs (real centre row)?
  bool obs_sym = true;
  {
    double mx = 0.0, res = 0.0;
    for (size_t i = 0; i < (size_t)2 * n * Np; ++i) mx = std::max(mx, std::fabs(ts->h_m1o[i]));
    for (int v = 0; v < (n + 1) / 2; ++v)
      for (int y = 0; y < Np; ++y) {
        const double* a = &ts->h_m1o[2 * ((size_t)v * Np + y)];
        const double* b = &ts->h_m1o[2 * ((size_t)(n - 1 - v) * Np + y)];
        res = std::max(res, std::max(std::fabs(a[0] - b[0]), std::fabs(a[1] + b[1])));
      }
    obs_sym = res <= 1e-12 * mx;
  }
  ts->sym = obs_sym && ts->g_real && getenv("AOG_FUSED_GENERIC") == nullptr;
  {
    std::vector<double> ph((size_t)2 * AOG_MAX_LP, 0.0);
    for (int j = 0; j < J; ++j) {
      const double th = ts->sym ? ts->theta[j] : 0.0;
      const double pr = ts->h_lpphase[2 * j], pi = ts->h_lpphase[2 * j + 1];
      ph[2 * j] = pr * std::cos(th) - pi * std::sin(th);
      ph[2 * j + 1] = pr * std::sin(th) + pi * std::cos(th);
    }
    AOG_CUDA(cudaMemcpy(ts->lpphase_f, ph.data(), ph.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  if (ts->sym) {
    const int NF = FK_NF(n), np2 = n / 2, nc = n & 1;
    std::vector<float> g((size_t)Np * Np * NF, 0.f);
    for (int y = 0; y < Np; ++y)
      for (int x = 0; x < Np; ++x) {
        const double a = ts->h_ap[(size_t)y * Np + x] != 0.0 ? 1.0 : 0.0;
        float* rec = &g[(((size_t)x * (Np / 16) + y / 16) * 16 + y % 16) * NF];
        for (int v = 0; v < np2; ++v) {
          rec[2 * v] = (float)(a * ts->h_m1o[2 * ((size_t)v * Np + y)]);
          rec[2 * v + 1] = (float)(a * ts->h_m1o[2 * ((size_t)v * Np + y) + 1]);
        }
        if (nc) rec[2 * np2] = (float)(a * ts->h_m1o[2 * ((size_t)np2 * Np + y)]);
        for (int j = 0; j < J; ++j) {
          const size_t src = 2 * (((size_t)j * Np + y) * Np + x);
          const double re = ts->h_G[src] * std::cos(ts->theta[j]) + ts->h_G[src + 1] * std::sin(ts->theta[j]);
          rec[2 * np2 + nc + j] = (float)(a * re / ts->gfib_scale);
        }
        rec[2 * np2 + nc + FK_JT] = (float)a;
      }
    AOG_CUDA(cudaMemcpy(ts->gfib, g.data(), g.size() * sizeof(float), cudaMemcpyHostToDevice));
    ts->have_gfib = true;
    return AOG_OK;
  }
  std::vector<float2> g((size_t)Np * Np * NT, make_float2(0.f, 0.f));
  for (int y = 0; y < Np; ++y)
    for (int x = 0; x < Np; ++x) {
      const double a = ts->h_ap[(size_t)y * Np + x] != 0.0 ? 1.0 : 0.0;
      float2* rec = &g[(((size_t)x * (Np / 16) + y / 16) * 16 + y % 16) * NT];
      for (int v = 0; v < n; ++v)
        rec[v] = make_float2((float)(a * ts->h_m1o[2 * ((size_t)v * Np + y)]), (float)(a * ts->h_m1o[2 * ((size_t)v * Np + y) + 1]));
      for (int j = 0; j < J; ++j) {
        const size_t src = 2 * (((size_t)j * Np + y) * Np + x);
        rec[n + j] = make_float2((float)(a * ts->h_G[src] / ts->gfib_scale), (float)(a * ts->h_G[src + 1] / ts->gfib_scale));
      }
      rec[n + FK_JT] = make_float2((float)a, 0.f);
    }
  AOG_CUDA(cudaMemcpy(ts->gfib, g.data(), g.size() * sizeof(float2), cudaMemcpyHostToDevice));
  ts->have_gfib = true;
  return AOG_OK;
}
}  // namespace

int aog_tensor_sh_table(aog_env* env, int which, const void* host);   // sh_tensor.cuh

int aog_tensor_table_updated(aog_env* env, int which, const void* host) {
  TensorState* ts = env->tensor.get();
  const aog_config& c = env->cfg;
  const int Np = c.num_pupil_pixels, Nf = c.num_focal_pixels;     // the tensor-precision branches below run at 240 / 128 only
  if (which >= AOG_TABLE_SH_MLA_PHASE && which <= AOG_TABLE_SH_ACT0) return aog_tensor_sh_table(env, which, host);
  if (ts->fused && which == AOG_TABLE_LP_PHASE) {
    const double* m = static_cast<const double*>(host);
    ts->h_lpphase.assign(m, m + (size_t)2 * c.num_lp_modes);
    ts->have_lpphase = true;
    return build_fused_records(env, ts);
  }
  if (ts->fused && (which == AOG_TABLE_MFT_FIB_1 || which == AOG_TABLE_MFT_FIB_2 || which == AOG_TABLE_LP_MODES_W)) {
    const double* m = static_cast<const double*>(host);
    if (which == AOG_TABLE_MFT_FIB_1) { ts->h_m1.assign(m, m + (size_t)2 * Nf * Np); ts->have_m1 = true; }
    if (which == AOG_TABLE_MFT_FIB_2) { ts->h_m2.assign(m, m + (size_t)2 * Np * Nf); ts->have_m2 = true; }
    if (which == AOG_TABLE_LP_MODES_W) { ts->h_lp.assign(m, m + (size_t)c.num_lp_modes * env->NF2); ts->have_lp = true; }
    if (ts->have_m1 && ts->have_m2 && ts->have_lp) {
      int rc = build_backprojected_modes(env, ts);
      if (rc) return rc;
      return build_fused_records(env, ts);
    }
    return AOG_OK;
  }
  if (which == AOG_TABLE_MFT_FIB_1) {
    // M1 [Nf][Np] complex, every entry of modulus w (the pupil grid weight): factor it out.
    const double* m = static_cast<const double*>(host);
    const double w = std::hypot(m[0], m[1]);
    ts->pupil_weight = w;
    std::vector<double> a((size_t)256 * TC_K);
    for (int v = 0; v < Nf; ++v)
      for (int y = 0; y < Np; ++y) {
        const double re = m[2 * ((size_t)v * Np + y)] / w, im = m[2 * ((size_t)v * Np + y) + 1] / w;
        // contraction order of stage 1: block y / 16 = [16 y against Er | the same 16 y against Ei]
        const int kr = (y >> 4) * 32 + (y & 15), ki = kr + 16;
        a[(size_t)v * TC_K + kr] = re;              // Tr rows:  M1r . Er - M1i . Ei
        a[(size_t)v * TC_K + ki] = -im;
        a[(size_t)(128 + v) * TC_K + kr] = im;      // Ti rows:  M1i . Er + M1r . Ei
        a[(size_t)(128 + v) * TC_K + ki] = re;
      }
    int rc = upload_split(env, a, ts->A1_hi, ts->A1_lo);
    if (rc) return rc;
    ts->have_m1 = true;
  } else if (which == AOG_TABLE_MFT_FIB_2) {
    // M2 [Np][Nf] complex (unit modulus).  Operand rows n = (u | 128 + u), K = (x | 240 + x):
    //   Fr[u] = sum_x Tr[x] M2r[x][u] - Ti[x] M2i[x][u];   Fi[u] = sum_x Tr[x] M2i[x][u] + Ti[x] M2r[x][u]
    const double* m = static_cast<const double*>(host);
    std::vector<double> b((size_t)256 * TC_K);
    for (int x = 0; x < Np; ++x)
      for (int u = 0; u < Nf; ++u) {
        const double re = m[2 * ((size_t)x * Nf + u)], im = m[2 * ((size_t)x * Nf + u) + 1];
        // operand rows: CTA r = u / 64 owns rows [128 r, 128 r + 128) = [Fr rows of its 64 u | Fi rows of its 64 u]
        const size_t rr = (size_t)(u / 64) * 128 + u % 64, ri = rr + 64;
        b[rr * TC_K + x] = re;
        b[rr * TC_K + Np + x] = -im;
        b[ri * TC_K + x] = im;
        b[ri * TC_K + Np + x] = re;
      }
    int rc = upload_split(env, b, ts->B2_hi, ts->B2_lo);
    if (rc) return rc;
    ts->have_m2 = true;
  } else if (which == AOG_TABLE_LP_MODES_W) {
    const double* m = static_cast<const double*>(host);
    const size_t cnt = (size_t)c.num_lp_modes * env->NF2;
    double mx = 0.0;
    for (size_t i = 0; i < cnt; ++i) mx = std::max(mx, std::fabs(m[i]));
    if (mx == 0.0) mx = 1.0;
    ts->lpw_scale = mx;
    // stored transposed ([j][u][v]): the stage-2 accumulator is F^T (lane = focal column u)
    std::vector<float> f(cnt);
    for (int j = 0; j < c.num_lp_modes; ++j)
      for (int v = 0; v < Nf; ++v)
        for (int u = 0; u < Nf; ++u)
          f[((size_t)j * Nf + u) * Nf + v] = (float)(m[((size_t)j * Nf + v) * Nf + u] / mx);
    AOG_CUDA(cudaMemcpy(ts->lpw, f.data(), cnt * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<float> g(cnt);
    const int J = c.num_lp_modes;
    for (int j = 0; j < J; ++j)
      for (int v = 0; v < Nf; ++v)
        for (int u = 0; u < Nf; ++u) {
          const size_t tile = ((size_t)(u / 64) * (Nf / 16) + v / 16) * J + j;
          g[((tile * 4 + (v / 4) % 4) * 64 + u % 64) * 4 + (v & 3)] = (float)(m[((size_t)j * Nf + v) * Nf + u] / mx);
        }
    AOG_CUDA(cudaMemcpy(ts->lpwr, g.data(), cnt * sizeof(float), cudaMemcpyHostToDevice));
    ts->have_lp = true;
  } else if (which == AOG_TABLE_DM_MODES) {
    // modes [K][y][x] FP64 -> GEMM B operand [x][y][KPAD] split fp16 (k contiguous, zero padded)
    const double* m = static_cast<const double*>(host);
    const int kp = ts->kpad;
    std::vector<double> f((size_t)env->P * kp, 0.0);
    for (int k = 0; k < c.num_modes; ++k)
      for (int y = 0; y < Np; ++y)
        for (int x = 0; x < Np; ++x) f[((size_t)x * Np + y) * kp + k] = m[((size_t)k * Np + y) * Np + x];
    int rc = upload_split(env, f, ts->modesK_hi, ts->modesK_lo);
    if (rc) return rc;
    ts->have_modes = true;
  } else if (which == AOG_TABLE_APERTURE) {
    const double* m = static_cast<const double*>(host);
    std::vector<uint16_t> bits((size_t)Np * (Np / 16), 0);
    for (int y = 0; y < Np; ++y)
      for (int x = 0; x < Np; ++x)
        if (m[(size_t)y * Np + x] != 0.0) bits[(size_t)x * (Np / 16) + y / 16] |= (uint16_t)(1u << (y % 16));
    AOG_CUDA(cudaMemcpy(ts->apmask, bits.data(), bits.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    ts->have_ap = true;
    if (ts->fused) { ts->h_ap.assign(m, m + (size_t)Np * Np); return build_fused_records(env, ts); }
  } else if (which == AOG_TABLE_MFT_OBS_1) {
    const double* m = static_cast<const double*>(host);   // [n][Np] complex
    std::vector<float2> f((size_t)c.obs_dim * Np);
    for (size_t i = 0; i < f.size(); ++i) f[i] = make_float2((float)m[2 * i], (float)m[2 * i + 1]);
    AOG_CUDA(cudaMemcpy(ts->m1o32, f.data(), f.size() * sizeof(float2), cudaMemcpyHostToDevice));
    ts->have_m1o = true;
    if (ts->fused) { ts->h_m1o.assign(m, m + (size_t)2 * c.obs_dim * Np); return build_fused_records(env, ts); }
  } else if (which == AOG_TABLE_MFT_OBS_2) {
    const double* m = static_cast<const double*>(host);   // [Np][n] complex -> [n][Np]
    const int n = c.obs_dim;
    std::vector<double> f((size_t)2 * n * Np);
    for (int x = 0; x < Np; ++x)
      for (int u = 0; u < n; ++u) {
        f[2 * ((size_t)u * Np + x)] = m[2 * ((size_t)x * n + u)];
        f[2 * ((size_t)u * Np + x) + 1] = m[2 * ((size_t)x * n + u) + 1];
      }
    AOG_CUDA(cudaMemcpy(ts->m2oT, f.data(), f.size() * sizeof(double), cudaMemcpyHostToDevice));
    ts->have_m2o = true;
  }
  return AOG_OK;
}

int aog_tensor_screens_updated(aog_env* env) {
  TensorState* ts = env->tensor.get();
  const int Np = env->cfg.num_pupil_pixels, B = env->cfg.num_envs;
  const double pi = 3.14159265358979323846;
  const size_t total = (size_t)((B + 127) / 128) * 4 * Np * (Np / 16) * 512;
  k_screens_to_tiles<<<(unsigned)((total + 255) / 256), 256>>>(env->screens, ts->hwt, Np, B, total,
                                                              1.0 / (env->cfg.wavelength_wfs * pi), nullptr);
  AOG_LAUNCH_CHECK();
  AOG_CUDA(cudaDeviceSynchronize());
  return AOG_OK;
}

int aog_tensor_rescale_screens(aog_env* env, const double* factor_dev, cudaStream_t st) {
  TensorState* ts = env->tensor.get();
  const int Np = env->cfg.num_pupil_pixels, B = env->cfg.num_envs;
  const double pi = 3.14159265358979323846;
  const size_t total = (size_t)((B + 127) / 128) * 4 * Np * (Np / 16) * 512;
  k_screens_to_tiles<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(env->screens, ts->hwt, Np, B, total,
                                                                     1.0 / (env->cfg.wavelength_wfs * pi), factor_dev);
  AOG_LAUNCH_CHECK();
  return AOG_OK;
}

// Debug read-back (tests): the split-fp16 intermediates of the LAST chunk processed, recombined
// hi + lo and returned in the FP64 path's conventions.
//   which = AOG_FIELD_TC_PUPIL : pupil field [y][x] complex (unit modulus x aperture)
//   which = AOG_FIELD_TC_STAGE1: stage-1 product [v][x] complex (unit-modulus twiddles)
int aog_tensor_get_field(aog_env* env, int which, int env_in_chunk, double* host_out, size_t count) {
  TensorState* ts = env->tensor.get();
  if (!ts || ts->fused) AOG_FAIL(AOG_ERR_STATE, "handle has no matrix-Fourier-transform GEMM stages");
  if (env_in_chunk < 0 || env_in_chunk >= env->chunk) AOG_FAIL(AOG_ERR_INVALID, "env index outside the chunk");
  if (which == AOG_FIELD_TC_PUPIL) {          // phi [y / 16][x][16] radians -> out [y][x] = aperture exp(i phi)
    if (count != (size_t)2 * TC_NP * TC_NP) AOG_FAIL(AOG_ERR_INVALID, "count");
    std::vector<float> ph((size_t)TC_NP * TC_NP);
    std::vector<uint16_t> ap((size_t)TC_NP * (TC_NP / 16));
    AOG_CUDA(cudaMemcpy(ph.data(), ts->phi + (size_t)env_in_chunk * ph.size(), ph.size() * sizeof(float), cudaMemcpyDeviceToHost));
    AOG_CUDA(cudaMemcpy(ap.data(), ts->apmask, ap.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    for (int x = 0; x < TC_NP; ++x)
      for (int y = 0; y < TC_NP; ++y) {
        const bool lit = (ap[(size_t)x * (TC_NP / 16) + y / 16] >> (y % 16)) & 1;
        const double a = (double)ph[((size_t)(y / 16) * TC_NP + x) * 16 + y % 16];
        host_out[2 * ((size_t)y * TC_NP + x)] = lit ? std::cos(a) : 0.0;
        host_out[2 * ((size_t)y * TC_NP + x) + 1] = lit ? std::sin(a) : 0.0;
      }
    return AOG_OK;
  }
  if (count != (size_t)2 * 128 * TC_NP) AOG_FAIL(AOG_ERR_INVALID, "count");
  const size_t nel = (size_t)128 * TC_K;
  std::vector<__half> hi(nel), lo(nel);
  AOG_CUDA(cudaMemcpy(hi.data(), ts->T_hi + (size_t)env_in_chunk * nel, nel * sizeof(__half), cudaMemcpyDeviceToHost));
  AOG_CUDA(cudaMemcpy(lo.data(), ts->T_lo + (size_t)env_in_chunk * nel, nel * sizeof(__half), cudaMemcpyDeviceToHost));
  auto val = [&](size_t i) { return (double)__half2float(hi[i]) + (double)__half2float(lo[i]); };
  for (int v = 0; v < 128; ++v)                 // stored [v][k = x | 240 + x]  ->  out [v][x]
    for (int x = 0; x < TC_NP; ++x) {
      host_out[2 * ((size_t)v * TC_NP + x)] = val((size_t)v * TC_K + x);
      host_out[2 * ((size_t)v * TC_NP + x) + 1] = val((size_t)v * TC_K + TC_NP + x);
    }
  return AOG_OK;
}

// AO_env.py:115-120 for every env, with the DM-GEMM operand packed in the same kernel.  Returns AOG_ERR_UNSUPPORTED
// (and launches nothing) when the handle runs more than one chunk or the Gram matrix does not fit shared memory.
int aog_tensor_actuators(aog_env* env, const void* actions_dev, int act_dtype, cudaStream_t st) {
  TensorState* ts = env->tensor.get();
  const aog_config& c = env->cfg;
  const int B = c.num_envs, K = c.num_modes;
  const size_t shm = ((size_t)K * K + 8 * (size_t)K) * sizeof(double);
  if (!ts || B > env->chunk || shm > 48 * 1024) return AOG_ERR_UNSUPPORTED;
  const int grid = std::min(cdiv(B, 8), 4 * ts->num_sms);
  const double target = 0.1 * c.wavelength_sci, pscale = 4.0 / c.wavelength_wfs;
  if (act_dtype == AOG_DTYPE_F32)
    k_actuators_pack<float><<<grid, 256, shm, st>>>((const float*)actions_dev, env->t_gram, env->act, ts->act_hi, ts->act_lo,
                                                    B, K, ts->kpad, c.sh_operation, target, pscale);
  else
    k_actuators_pack<double><<<grid, 256, shm, st>>>((const double*)actions_dev, env->t_gram, env->act, ts->act_hi,
                                                     ts->act_lo, B, K, ts->kpad, c.sh_operation, target, pscale);
  AOG_LAUNCH_CHECK();
  ts->packed_valid = true;
  return AOG_OK;
}

void aog_tensor_annotate_error(aog_env* env) {
  TensorState* ts = env ? env->tensor.get() : nullptr;
  if (!ts || !ts->err_flag_host) return;
  const int flag = *(volatile int*)ts->err_flag_host;
  if (flag) env->err += " [tensor pipeline barrier timeout, code " + std::to_string(flag) + ": the kernel trapped, this process's CUDA context is no longer usable]";
}

int aog_tensor_check(aog_env* env) {
  TensorState* ts = env->tensor.get();
  if (!ts) return AOG_OK;
  const int flag = ts->err_flag_host ? *(volatile int*)ts->err_flag_host : 0;
  if (flag) AOG_FAIL(AOG_ERR_CUDA, "tensor pipeline barrier timeout, code " + std::to_string(flag) +
                                       " (the kernel trapped: this process's CUDA context is no longer usable)");
  return AOG_OK;
}

namespace {
template <bool STREHL, int NOBS, int MODE, int NP = TC_NP>
int launch_phase(aog_env* env, TensorState* ts, const FieldParams& p, int grid, cudaStream_t st) {
  constexpr bool FUSED = MODE == 1 || MODE == 2;
  constexpr int smem = FK_STAGES * FK_STAGE_BYTES + FK_PF_BYTES(NOBS, MODE) + 1024 + FK_AUX_BAR +
                       (FUSED ? 1 + FK_JT : 1) * FK_PARTS * 128 * (int)sizeof(double2) +
                       (FUSED ? 0 : NOBS * NP * (int)sizeof(float2) + NP * (NP / 16) * (int)sizeof(uint16_t)) +
                       2 * NP * FK_NSEG(NP);
  static_assert(smem <= 227 * 1024, "shared memory of the phase kernel");
  static std::atomic<bool> configured_on[64];   // function attributes are per device: one flag per device ordinal
  std::atomic<bool>& configured = configured_on[env->cfg.device & 63];
  if (!configured.load(std::memory_order_acquire)) {
    AOG_CUDA(cudaFuncSetAttribute(k_dm_phase_tc<STREHL, NOBS, MODE, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured.store(true, std::memory_order_release);
  }
  k_dm_phase_tc<STREHL, NOBS, MODE, NP><<<grid, FK_THREADS, smem, st>>>(ts->tmAct_hi, ts->tmAct_lo, ts->tmModes_hi, ts->tmModes_lo,
                                                                        ts->tmHwt, p);
  AOG_LAUNCH_CHECK();
  return AOG_OK;
}
template <bool STREHL, int MODE>
int launch_phase_n(aog_env* env, TensorState* ts, const FieldParams& p, int n, int grid, cudaStream_t st) {
  const int Np = env->cfg.num_pupil_pixels;
  if (Np != TC_NP) {
    // the pupil-grid axis of BASELINE configs[4]: fused kernels for 128^2, 256^2 and 512^2 pupils, detectors 2x2 and 5x5
    if constexpr (MODE == 1 || MODE == 2) {
      if (Np == 128 && n == 2) return launch_phase<STREHL, 2, MODE, 128>(env, ts, p, grid, st);
      if (Np == 128 && n == 5) return launch_phase<STREHL, 5, MODE, 128>(env, ts, p, grid, st);
      if (Np == 256 && n == 2) return launch_phase<STREHL, 2, MODE, 256>(env, ts, p, grid, st);
      if (Np == 256 && n == 5) return launch_phase<STREHL, 5, MODE, 256>(env, ts, p, grid, st);
      if (Np == 512 && n == 2) return launch_phase<STREHL, 2, MODE, 512>(env, ts, p, grid, st);
      if (Np == 512 && n == 5) return launch_phase<STREHL, 5, MODE, 512>(env, ts, p, grid, st);
    }
    AOG_FAIL(AOG_ERR_UNSUPPORTED, "fused kernels for pupils other than 240^2 are built for 128^2 / 256^2 / 512^2 with obs_dim 2 or 5");
  }
  switch (n) {
    case 1: return launch_phase<STREHL, 1, MODE>(env, ts, p, grid, st);
    case 2: return launch_phase<STREHL, 2, MODE>(env, ts, p, grid, st);
    case 3: return launch_phase<STREHL, 3, MODE>(env, ts, p, grid, st);
    case 4: return launch_phase<STREHL, 4, MODE>(env, ts, p, grid, st);
    case 5: return launch_phase<STREHL, 5, MODE>(env, ts, p, grid, st);
    case 6: return launch_phase<STREHL, 6, MODE>(env, ts, p, grid, st);
    case 7: return launch_phase<STREHL, 7, MODE>(env, ts, p, grid, st);
    case 8: return launch_phase<STREHL, 8, MODE>(env, ts, p, grid, st);
  }
  AOG_FAIL(AOG_ERR_UNSUPPORTED, "obs_dim");
}
template <bool STREHL>
int launch_small(aog_env* env, const SmallParams& sp, int n, cudaStream_t st) {
  const int grid = cdiv(sp.Np, sp.ipc);
  switch (n) {
    case 1: k_small_fused<STREHL, 1><<<grid, 256, 0, st>>>(sp); break;
    case 2: k_small_fused<STREHL, 2><<<grid, 256, 0, st>>>(sp); break;
    case 3: k_small_fused<STREHL, 3><<<grid, 256, 0, st>>>(sp); break;
    case 4: k_small_fused<STREHL, 4><<<grid, 256, 0, st>>>(sp); break;
    case 5: k_small_fused<STREHL, 5><<<grid, 256, 0, st>>>(sp); break;
    case 6: k_small_fused<STREHL, 6><<<grid, 256, 0, st>>>(sp); break;
    case 7: k_small_fused<STREHL, 7><<<grid, 256, 0, st>>>(sp); break;
    case 8: k_small_fused<STREHL, 8><<<grid, 256, 0, st>>>(sp); break;
    default: AOG_FAIL(AOG_ERR_UNSUPPORTED, "obs_dim");
  }
  AOG_LAUNCH_CHECK();
  return AOG_OK;
}
// k_finalize_tcw<n, PARTS>: one warp per env, dynamic shared memory above 48 KB (opt-in once per device).
// PARTS = partial sums per contraction index in R4: FK_PARTS, or 2 FK_PARTS for the two column segments of a 512^2 pupil.
template <int N, int PARTS = FK_PARTS>
cudaError_t launch_finalize(int device, const FinalizeArgs& a, int nB, cudaStream_t st) {
  using Cfg = FinCfg<N, PARTS>;
  static_assert(Cfg::SMEM + Cfg::TAB_MAX <= 227 * 1024, "shared memory of k_finalize_tcw");
  static std::atomic<bool> configured_on[64];
  std::atomic<bool>& configured = configured_on[device & 63];
  if (!configured.load(std::memory_order_acquire)) {
    const cudaError_t e = cudaFuncSetAttribute(k_finalize_tcw<N, PARTS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               Cfg::SMEM + Cfg::TAB_MAX);
    if (e != cudaSuccess) return e;
    configured.store(true, std::memory_order_release);
  }
  if (a.Np > 512) return cudaErrorInvalidValue;
  k_finalize_tcw<N, PARTS><<<cdiv(nB, FIN_WARPS), FIN_WARPS * 32, Cfg::SMEM + N * a.Np * 16, st>>>(a, nB);
  return cudaSuccess;
}
}  // namespace

int aog_tensor_optics(aog_env* env, bool flat_dm, bool with_reward, const aog_outputs& out, cudaStream_t st) {
  TensorState* ts = env->tensor.get();
  const aog_config& c = env->cfg;
  if (!(ts->have_m1 && ts->have_m2 && ts->have_lp && ts->have_modes && ts->have_ap && ts->have_m2o && ts->have_m1o) ||
      (ts->fused && !ts->have_gfib))
    AOG_FAIL(AOG_ERR_STATE, "tensor path tables incomplete");
  const bool fused = ts->fused;
  (void)flat_dm;                         // the caller has already zeroed the actuators of a flattened mirror
  const int Np = c.num_pupil_pixels, n = c.obs_dim, K = c.num_modes, J = c.num_lp_modes, B = c.num_envs;
  const bool strehl = with_reward && c.rew_type == AOG_REW_STREHL_RATIO;
  const double2 norm = make_double2(c.mft_norm_re * c.amp_fiber, c.mft_norm_im * c.amp_fiber);
  const int nseg = FK_NSEG(Np), items_per_block = Np * nseg;      // phase-kernel work items: column segments
  int slot_ipc = 1;
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    if (env->timing) { AOG_CUDA(cudaEventRecord(env->evf.get(), st)); }
    {
      // actuators -> half-turns of DM phase per unit mode (2 k s / pi = 4 s / lambda), split fp16
      const int rows = cdiv(nB, 128) * 128;
      if (!ts->packed_valid) {
        k_act_pack<<<cdiv(rows * ts->kpad, 256), 256, 0, st>>>(env->act, ts->act_hi, ts->act_lo, K, ts->kpad, e0, nB,
                                                               rows, 4.0 / c.wavelength_wfs);
        AOG_LAUNCH_CHECK();
      }
      ts->packed_valid = false;                      // good for the one optics pass that follows k_actuators_pack
      FieldParams fp{};
      fp.num_envs = nB;
      fp.num_items = cdiv(nB, 128) * items_per_block;
      // an env block's items touch at most cdiv(items_per_block, items_per_cta) + 1 <= FK_SLOTS CTAs
      fp.items_per_cta = std::max(std::max(FK_MIN_ITEMS, cdiv(items_per_block, FK_SLOTS - 1)), cdiv(fp.num_items, ts->num_sms));
      fp.nkb = ts->kpad / 64;
      fp.col_origin = (int)env->cnt.column_origin;
      fp.env0 = e0;
      { const char* d = getenv("AOG_FK_DEBUG"); fp.dbg = d ? atoi(d) : 0; }
      fp.sci_ratio_q32 = (uint32_t)std::llround(c.wavelength_wfs / c.wavelength_sci * 4294967296.0);
      fp.apmask = ts->apmask; fp.m1o32 = ts->m1o32; fp.phi = ts->phi; fp.R4 = ts->R4;
      fp.strehl_part = env->strehl_part;
      fp.gfib = ts->gfib; fp.fib_part = ts->fib_part;
      fp.err_flag = ts->err_flag;
      const int grid = cdiv(fp.num_items, fp.items_per_cta);
      int rc;
      slot_ipc = fp.items_per_cta;            // k_finalize_tcw sums exactly the slots this launch writes
      const bool no_small = getenv("AOG_NO_SMALL") != nullptr;             // A/B switch and test hook: tensor cores for every batch size
      if (fused && ts->sym && B <= SMALL_MAX && !no_small && ts->kpad <= 128 && Np <= 256 && !fp.dbg) {
        SmallParams sp{};
        sp.B = nB; sp.Np = Np; sp.kpad = ts->kpad; sp.col_origin = fp.col_origin; sp.env0 = e0;
        sp.ipc = cdiv(Np, std::min(ts->num_sms, FK_SLOTS));
        sp.sci_ratio_q32 = fp.sci_ratio_q32;
        sp.hwt = ts->hwt; sp.apmask = ts->apmask; sp.gfib = reinterpret_cast<const float*>(ts->gfib.get());
        sp.act_hi = ts->act_hi; sp.act_lo = ts->act_lo; sp.m_hi = ts->modesK_hi; sp.m_lo = ts->modesK_lo;
        sp.R4 = ts->R4; sp.strehl_part = env->strehl_part; sp.fib_part = ts->fib_part;
        slot_ipc = sp.ipc;
        rc = strehl ? launch_small<true>(env, sp, n, st) : launch_small<false>(env, sp, n, st);
      } else
      if (fused && ts->sym) rc = strehl ? launch_phase_n<true, 2>(env, ts, fp, n, grid, st) : launch_phase_n<false, 2>(env, ts, fp, n, grid, st);
      else if (fused)       rc = strehl ? launch_phase_n<true, 1>(env, ts, fp, n, grid, st) : launch_phase_n<false, 1>(env, ts, fp, n, grid, st);
      else                  rc = strehl ? launch_phase_n<true, 0>(env, ts, fp, n, grid, st) : launch_phase_n<false, 0>(env, ts, fp, n, grid, st);
      if (rc) return rc;
    }
    if (env->timing) { AOG_CUDA(cudaEventRecord(env->ev0.get(), st)); }
    const int max_clusters = ts->num_sms / 2;
    int tc_dbg = 0;
    { const char* d = getenv("AOG_TC_DEBUG"); tc_dbg = d ? atoi(d) : 0; }
    if (!fused) {
      F1Params f1{};
      f1.num_items = nB;
      f1.apmask = ts->apmask;
      f1.dbg = tc_dbg; f1.err_flag = ts->err_flag;
      static std::atomic<bool> configured_on[64];
      std::atomic<bool>& configured = configured_on[c.device & 63];
      if (!configured.load(std::memory_order_acquire)) {
        AOG_CUDA(cudaFuncSetAttribute(k_field_mft1, cudaFuncAttributeMaxDynamicSharedMemorySize, F1_SMEM_BYTES));
        configured.store(true, std::memory_order_release);
      }
      k_field_mft1<<<2 * std::min(max_clusters, nB), F1_THREADS, F1_SMEM_BYTES, st>>>(ts->tmA1_hi, ts->tmA1_lo, ts->tmPhi,
                                                                                   ts->tmTout_hi, ts->tmTout_lo, f1);
      AOG_LAUNCH_CHECK();
    }
    if (env->timing) { AOG_CUDA(cudaEventRecord(env->evm.get(), st)); }
    if (with_reward && !fused) {
      TcParams p{};
      p.num_envs = nB;
      p.err_flag = ts->err_flag;
      p.dbg = tc_dbg;
      p.T_hi = ts->T_hi; p.T_lo = ts->T_lo;
      p.lpw = ts->lpw; p.lpwr = ts->lpwr; p.coef_raw = ts->coef4; p.J = J;
      p.num_items = (nB + 1) / 2;
      if (J <= 3)
        k_mft2<3><<<2 * std::min(max_clusters, p.num_items), M2_THREADS, M2_SMEM_BYTES, st>>>(
            ts->tmB2_hi, ts->tmB2_lo, ts->tmT128_hi, ts->tmT128_lo, p);
      else
        k_mft2<AOG_MAX_LP><<<2 * std::min(max_clusters, p.num_items), M2_THREADS, M2_SMEM_BYTES, st>>>(
            ts->tmB2_hi, ts->tmB2_lo, ts->tmT128_hi, ts->tmT128_lo, p);
      AOG_LAUNCH_CHECK();
    }
    if (env->timing) { AOG_CUDA(cudaEventRecord(env->ev1.get(), st)); env->ev_valid = true; }
    FinalizeArgs a{};
    a.R4 = ts->R4; a.m1o = ts->m2oT;
    {
      // coef holds the raw projection sums (re, im): scale = norm * amp * pupil weight * table scale
      const double sc = fused ? c.amp_fiber * ts->gfib_scale : c.amp_fiber * ts->pupil_weight * ts->lpw_scale;
      a.coef_scale = make_double2(c.mft_norm_re * sc, c.mft_norm_im * sc);
      a.coef_is_raw = fused ? 3 : 2;
      a.fib_part = ts->fib_part; a.fib_slots = FK_SLOTS; a.fib_stride = FK_JT;
    } a.coef4 = ts->coef4; a.lpphase = fused ? ts->lpphase_f : env->t_lpphase; a.lpgram = env->t_lpgram;
    a.strehl_part = env->strehl_part; a.strehl_blocks = FK_SLOTS;
    a.slot_ipc = slot_ipc; a.slot_items = items_per_block;
    a.act = env->act + (size_t)e0 * K; a.K = K;      // (a flattened mirror has zero, not NaN, actuators)
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
    if (nseg == 2) {
      if (n == 2) AOG_CUDA((launch_finalize<2, 2 * FK_PARTS>(c.device, a, nB, st)));
      else if (n == 5) AOG_CUDA((launch_finalize<5, 2 * FK_PARTS>(c.device, a, nB, st)));
      else AOG_FAIL(AOG_ERR_UNSUPPORTED, "fused kernels for 512^2 pupils are built for obs_dim 2 or 5");
    } else switch (n) {
      case 1: AOG_CUDA(launch_finalize<1>(c.device, a, nB, st)); break;
      case 2: AOG_CUDA(launch_finalize<2>(c.device, a, nB, st)); break;
      case 3: AOG_CUDA(launch_finalize<3>(c.device, a, nB, st)); break;
      case 4: AOG_CUDA(launch_finalize<4>(c.device, a, nB, st)); break;
      case 5: AOG_CUDA(launch_finalize<5>(c.device, a, nB, st)); break;
      case 6: AOG_CUDA(launch_finalize<6>(c.device, a, nB, st)); break;
      case 7: AOG_CUDA(launch_finalize<7>(c.device, a, nB, st)); break;
      default: AOG_CUDA(launch_finalize<8>(c.device, a, nB, st)); break;
    }
    AOG_LAUNCH_CHECK();
  }
  return AOG_OK;
}

#include "sh_tensor.cuh"
