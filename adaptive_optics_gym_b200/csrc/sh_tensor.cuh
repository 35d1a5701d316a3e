// Shack-Hartmann integrator on the tensor cores (AOG_PRECISION_TENSOR / AOG_PRECISION_FUSED), sm_100a only.
// Included by tensor_path.cu (it uses that file's PTX wrappers, tensor-map helpers and TensorState).
//
// Reference: AOEnv.SH_step (gym_AO/envs/AO_env.py:254-290) -- atmosphere + the integrator's own mirror (:263-266),
// magnifier + micro-lens array + Fresnel propagation to the lenslet focal plane (:269, hcipy
// SquareShackHartmannWavefrontSensorOptics), camera image x dt and photon noise (:272-274), flux-weighted centroids
// per selected lenslet (:277-279), leaky integrator a <- 0.99 a - 0.3 R slopes (:282-285).
//
// The optics between the pupil and the camera is the separable linear map E_out = C (m o E) C^T: C is the Fresnel
// operator (2x zero-padded angular-spectrum FFT, cropped) and m = exp(i mla_phase) the micro-lens phase, which is
// separable too (m[y][x] = m_y[y] m_x[x]), so E_out = C1 E C2^T with C1 = C diag(m_y), C2 = C diag(m_x).  On hcipy's
// symmetric grids C1 and C2 are centrosymmetric: they act separately on the even and the odd part of a vector, and
// the product splits into four (N/2)^3 blocks (half the flops, exact):
//
//   E_pq[i][x] = E[i][x] + p E[N-1-i][x] + q E[i][N-1-x] + p q E[N-1-i][N-1-x]          (p, q = +-1; i, x < N/2)
//   Y_pq = C1_p E_pq,   G_pq = Y_pq C2_q^T,   F[i][u] = G++ + G+- + G-+ + G--  (and the three mirror images with signs)
//
// Five kernels per chunk of environments:
//   k_dm_phase_tc<.., MODE 3>  (tensor_path.cu) DM surface of the SH mirror as a tcgen05 GEMM + atmosphere -> phase (FP32)
//   k_sh_fold      phase -> unit-modulus field (MUFU sincos, aperture) -> the four parity-folded blocks, split fp16,
//                  in the K-major layout the first product streams
//   k_sh_gemm<1>   Y_pq = C1_p E_pq      tcgen05.mma cta_group::2 kind::f16 (M = 256 over a CTA pair: Yr | Yi rows)
//   k_sh_gemm<2>   G_pq = Y_pq C2_q^T    (M = 256: the rows of the p = + | p = - block, N = Gr | Gi columns)
//   k_sh_camera_tc unfold, |.|^2 x dt, photon noise (Philox, FP32 samplers), centroids, slopes, integrator
//
// k_sh_gemm: a cluster (CTA pair) is dedicated to ONE parity, so its constant operand (the real embedding of C_p,
// split fp16 hi + lo, 128 KB per CTA) is loaded into shared memory once and stays there; only the per-environment
// operand streams (TMA ring, 16 KB per K block per CTA).  The accumulator (128 lanes x 256 columns FP32) is double
// buffered in TMEM, so the epilogue of one item runs under the MMAs of the next.  Every product is three MMAs
// hi.lo + lo.hi + hi.hi into ONE accumulator (the separate correction accumulator of k_mft2 is traded for the
// second buffer: the centroid is a ratio of sums of the image, in which the accumulation bias cancels).
// Dimensions are padded 120 -> 128 (M, N) and 240 -> 256 (K): tiles stay aligned to the 16-column epilogue chunks.

namespace {

constexpr int SH_NH = TC_NP / 2;                     // 120: folded grid size
constexpr int SH_HP = 128;                           // ... padded
constexpr int SH_K = 2 * SH_HP;                      // 256: real-embedded contraction length [re | im], padded
constexpr int SH_NKB = SH_K / KB;                    // 8 K blocks of [16 re | 16 im]
constexpr int SG_STAGES = 4;
constexpr int SG_RES_BYTES = SH_NKB * 2 * A_TILE;    // 128 KB: resident operand, per K block [hi 8 KB][lo 8 KB]
constexpr int SG_STAGE_BYTES = 2 * A_TILE;           // 16 KB: streamed operand, [hi 8 KB][lo 8 KB]
constexpr int SG_OUT_BUFS = 2;
constexpr int SG_EPI_BYTES = 2 * SG_OUT_BUFS * 2 * M2_OUT_TILE;      // 32 KB: per column half, ring of (hi, lo) store tiles
constexpr int SG_EPI_WARPS = 8;
// warp 0 TMA, warp 1 MMA, warps 4-11 epilogue; warps 2, 3 and 12-15 are idle.  Fewer threads raise the register cap
// and change the generated code: a performance question of its own.
constexpr int SG_THREADS = 512;
constexpr int SG_SMEM_BYTES = SG_RES_BYTES + SG_STAGES * SG_STAGE_BYTES + SG_EPI_BYTES + 1024 /*align*/ + 1024 /*barriers*/;
static_assert(SG_SMEM_BYTES <= 232448, "k_sh_gemm shared memory");

struct ShGemmParams {
  int num_envs;          // environments in this chunk: items of each parity
  float* G;              // STAGE 2 output: [env][p][q][128 i'][re 128 u | im 128 u] FP32
  int dbg;               // AOG_SH_DEBUG bits (tuning only): 1 no MMA, 4 no epilogue work
  int* err_flag;
};

// 256-bit stores (sm_100): one instruction writes a whole 32-byte sector per lane
__device__ __forceinline__ void st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}

// STAGE 1: resident = A (M side: rows [Yr(i') | Yi(i')] of C1_parity, parity = p), streamed = B (N side: the folded
//          field E_{p,q}, CTA r stages the block q = r); D lanes = i', columns = (q, x).  Epilogue: split fp16 ->
//          YB[env][q][p][i'][K = (x / 16) 32 + x % 16 + 16 (rank = im)] through swizzled tiles and TMA stores.
// STAGE 2: resident = B (N side: rows [Gr(u) | Gi(u)] of C2_parity, parity = q; CTA r holds re | im), streamed = A
//          (M side: Y_{p,q}, CTA r stages p = r); D lanes = i' (of block p = rank), columns = (re | im, u).
//          Epilogue: FP32 -> G[env][p][q][i'][re | im][u].
template <int STAGE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SG_THREADS, 1)
k_sh_gemm(const __grid_constant__ CUtensorMap tmR_hi, const __grid_constant__ CUtensorMap tmR_lo,
          const __grid_constant__ CUtensorMap tmS_hi, const __grid_constant__ CUtensorMap tmS_lo,
          const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo, const ShGemmParams p) {
  constexpr uint32_t TX_BYTES = 2 * SG_STAGE_BYTES;                   // both CTAs' tiles complete on the leader's barrier
  constexpr uint32_t IDESC = umma_idesc_f16(256, 2 * SH_HP);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* res = base;                                                // resident operand
  uint8_t* ring = res + SG_RES_BYTES;                                 // streamed operand ring
  uint8_t* epi = ring + SG_STAGES * SG_STAGE_BYTES;                   // STAGE 1 store tiles
  uint64_t* full = reinterpret_cast<uint64_t*>(epi + SG_EPI_BYTES);
  uint64_t* empty = full + SG_STAGES;
  uint64_t* res_full = empty + SG_STAGES;
  uint64_t* tmem_full = res_full + 1;                                 // [2]
  uint64_t* tmem_empty = tmem_full + 2;                               // [2] (used in the leader only)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int parity = cluster_id & 1;                                  // the cluster's resident table: even | odd part
  const int first = cluster_id >> 1, stride = num_clusters >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmR_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmR_lo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmS_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmS_lo)) : "memory");
    for (int s = 0; s < SG_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(res_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * SG_EPI_WARPS); }
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
    // ===================== TMA producer (both CTAs; completion on the leader's barriers) =====================
    if (lane == 0) {
      {   // resident operand: my 128 rows of the parity's table, all K blocks, once
        if (rank == 0) mbar_expect_tx(res_full, 2 * SG_RES_BYTES);
        const uint32_t rb = mapa_rank(smem_u32(res_full), 0);
        const int row0 = parity * 256 + (int)rank * 128;
        for (int kb = 0; kb < SH_NKB; ++kb) {
          const uint32_t s0 = smem_u32(res + kb * SG_STAGE_BYTES);
          tma_load_2d_pair(s0, &tmR_hi, rb, kb * KB, row0);
          tma_load_2d_pair(s0 + A_TILE, &tmR_lo, rb, kb * KB, row0);
        }
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int item = first; item < p.num_envs; item += stride) {
        const int srow0 = ((item * 2 + parity) * 2 + (int)rank) * SH_HP;
        for (int kb = 0; kb < SH_NKB; ++kb) {
          mbar_wait<32>(&empty[stage], phase ^ 1, p.err_flag, 21);
          if (rank == 0) mbar_expect_tx(&full[stage], TX_BYTES);
          const uint32_t s0 = smem_u32(ring + stage * SG_STAGE_BYTES);
          const uint32_t fb = mapa_rank(smem_u32(&full[stage]), 0);
          tma_load_2d_pair(s0, &tmS_hi, fb, kb * KB, srow0);
          tma_load_2d_pair(s0 + A_TILE, &tmS_lo, fb, kb * KB, srow0);
          if (++stage == SG_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread of the leader CTA) =====================
    if (rank == 0 && lane == 0) {
      mbar_wait<32>(res_full, 0, p.err_flag, 22);
      tc_fence_after();
      int stage = 0, it = 0;
      uint32_t phase = 0;
      for (int item = first; item < p.num_envs; item += stride, ++it) {
        const int buf = it & 1;
        mbar_wait<32>(&tmem_empty[buf], ((it >> 1) & 1) ^ 1, p.err_flag, 23);
        tc_fence_after();
        const uint32_t d = tmem_base + buf * (2 * SH_HP);
        for (int kb = 0; kb < SH_NKB; ++kb) {
          mbar_wait(&full[stage], phase, p.err_flag, 24);
          tc_fence_after();
          const uint32_t s0 = smem_u32(ring + stage * SG_STAGE_BYTES);
          const uint32_t r0 = smem_u32(res + kb * SG_STAGE_BYTES);
          if (!(p.dbg & 1))
#pragma unroll
          for (int ks = 0; ks < KB / 16; ++ks) {
            const uint64_t r_hi = umma_desc_sw64(r0 + ks * 32), r_lo = umma_desc_sw64(r0 + A_TILE + ks * 32);
            const uint64_t s_hi = umma_desc_sw64(s0 + ks * 32), s_lo = umma_desc_sw64(s0 + A_TILE + ks * 32);
            const uint64_t a_hi = STAGE == 1 ? r_hi : s_hi, a_lo = STAGE == 1 ? r_lo : s_lo;
            const uint64_t b_hi = STAGE == 1 ? s_hi : r_hi, b_lo = STAGE == 1 ? s_lo : r_lo;
            tc_mma_f16_pair(d, a_hi, b_lo, IDESC, (kb | ks) != 0);     // corrections first, the main product last
            tc_mma_f16_pair(d, a_lo, b_hi, IDESC, 1);
            tc_mma_f16_pair(d, a_hi, b_hi, IDESC, 1);
          }
          tc_commit_pair(&empty[stage]);            // frees the slot in both CTAs when these MMAs retire
          if (++stage == SG_STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_pair(&tmem_full[buf]);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue: 8 warps, TMEM lane group = warp % 4, column half = (warp - 4) / 4 ========
    const int lg = warp & 3;
    const int half = (warp - 4) >> 2;
    const int row = lg * 32 + lane;                                   // i'
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
    const uint32_t tmem_empty_leader = mapa_rank(smem_u32(tmem_empty), 0);
    uint32_t out_seq = 0;
    int it = 0;
    for (int item = first; item < p.num_envs; item += stride, ++it) {
      const int buf = it & 1;
      mbar_wait(&tmem_full[buf], (it >> 1) & 1, p.err_flag, 25);
      tc_fence_after();
      const uint32_t acc_addr = lane_addr + buf * (2 * SH_HP) + half * SH_HP;
      if (!(p.dbg & 4)) {
        if constexpr (STAGE == 1) {
          // my column half is the block q = half; chunk i = its K block of stage 2 (16 x re | 16 x im: rank = im)
          uint8_t* ebuf = epi + half * (SG_OUT_BUFS * 2 * M2_OUT_TILE);
          const uint32_t sw = (uint32_t)((row >> 2) & 1);             // SWIZZLE_32B: 16-byte piece ^= address bit 7
          const int orow0 = ((item * 2 + half) * 2 + parity) * SH_HP;
#pragma unroll 1
          for (int i = 0; i < 8; ++i) {
            float v[16];
            tc_ld16(acc_addr + i * 16, v);
            tc_wait_ld();
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) split_pack2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
            uint8_t* t_hi = ebuf + (out_seq % SG_OUT_BUFS) * (2 * M2_OUT_TILE);
            uint8_t* t_lo = t_hi + M2_OUT_TILE;
            *reinterpret_cast<uint4*>(t_hi + row * 32 + ((0u ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(t_hi + row * 32 + ((1u ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
            *reinterpret_cast<uint4*>(t_lo + row * 32 + ((0u ^ sw) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            *reinterpret_cast<uint4*>(t_lo + row * 32 + ((1u ^ sw) << 4)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            // the store issued from the OTHER buffer one chunk ago must have left shared memory before anyone
            // writes that buffer again (next chunk): its issuer waits here, ahead of the barrier
            if (lg == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            if (half == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
            else           asm volatile("bar.sync 2, 128;" ::: "memory");
            if (lg == 0 && lane == 0) {
              tma_store_2d(&tmO_hi, smem_u32(t_hi), i * KB + (int)rank * 16, orow0);
              tma_store_2d(&tmO_lo, smem_u32(t_lo), i * KB + (int)rank * 16, orow0);
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            ++out_seq;
          }
        } else {
          // lane = row i' of block p = rank; my column half = re | im of G_{p,q}[i'][u], q = parity
          float* grow = p.G + ((size_t)((item * 2 + (int)rank) * 2 + parity) * SH_HP + row) * (2 * SH_HP) + half * SH_HP;
#pragma unroll 1
          for (int i = 0; i < 8; i += 2) {
            float v[32];
            tc_ld32(acc_addr + i * 16, v);
            tc_wait_ld();
            if (row < SH_NH) {
#pragma unroll
              for (int k = 0; k < 32; k += 8)
                if (i * 16 + k < SH_NH) st_global_v8(grow + i * 16 + k, v + k);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty_leader + buf * 8);   // this warp is done with the buffer
    }
    if (STAGE == 1 && lg == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores landed
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

// ----------------------------------------------------------------------------- phase -> folded field
// Thread = (fold column x < 120, 16-row chunk kb) of one environment: the phase at the four mirror images of its 16
// fold pixels (rows 16 kb + j and 239 - 16 kb - j, columns x and 239 - x) are four contiguous 64-byte runs of the
// phase buffer ([env][y / 16][x][16 y]).  Field = aperture x exp(i phase) (unit modulus: the amplitude is applied
// to the image), folded with the four sign pairs, split fp16, written as the [16 re | 16 im] piece of K block kb of
// row x in EB[env][p][q] (full 32-byte sectors).  Rows 120 ... 127 of block 7 are the zero padding of the contraction.
__global__ void __launch_bounds__(128)
k_sh_fold(const float* __restrict__ phi, const uint16_t* __restrict__ apmask, __half* __restrict__ e_hi,
          __half* __restrict__ e_lo, int nB) {
  constexpr int Np = TC_NP, NC = TC_NP / 16;
  const int x = threadIdx.x, kb = blockIdx.x, env = blockIdx.y;
  if (x >= SH_NH || env >= nB) return;
  const int ca = kb, cb = NC - 1 - kb, xa = x, xb = Np - 1 - x;
  const float* pe = phi + (size_t)env * Np * Np;
  float ph[4][16];
  const float4* src[4] = {reinterpret_cast<const float4*>(pe + ((size_t)ca * Np + xa) * 16),
                          reinterpret_cast<const float4*>(pe + ((size_t)cb * Np + xa) * 16),
                          reinterpret_cast<const float4*>(pe + ((size_t)ca * Np + xb) * 16),
                          reinterpret_cast<const float4*>(pe + ((size_t)cb * Np + xb) * 16)};
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 v = __ldg(src[m] + k);
      ph[m][4 * k] = v.x; ph[m][4 * k + 1] = v.y; ph[m][4 * k + 2] = v.z; ph[m][4 * k + 3] = v.w;
    }
  const uint32_t mk[4] = {apmask[xa * NC + ca], apmask[xa * NC + cb], apmask[xb * NC + ca], apmask[xb * NC + cb]};
  const int nvalid = kb == SH_NKB - 1 ? SH_NH - 16 * (SH_NKB - 1) : 16;   // block 7: fold rows 112 ... 119 only
  uint32_t oh[4][16], ol[4][16];      // [p q][8 re pairs | 8 im pairs] packed halves
#pragma unroll
  for (int j2 = 0; j2 < 8; ++j2) {
    float fre[4][2], fim[4][2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * j2 + h;
      float c[4], s[4];
      // m = 0: (row, col); 1: row-mirrored (index 15 - j of chunk cb); 2: column-mirrored; 3: both
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int jj = (m & 1) ? 15 - j : j;
        float sn, cs;
        __sincosf(ph[m][jj], &sn, &cs);
        const bool lit = ((mk[m] >> jj) & 1u) && j < nvalid;
        c[m] = lit ? cs : 0.f;
        s[m] = lit ? sn : 0.f;
      }
      // E_pq = E0 + p E1 + q E2 + p q E3;  block index (p < 0) * 2 + (q < 0)
      fre[0][h] = (c[0] + c[1]) + (c[2] + c[3]);  fim[0][h] = (s[0] + s[1]) + (s[2] + s[3]);
      fre[1][h] = (c[0] + c[1]) - (c[2] + c[3]);  fim[1][h] = (s[0] + s[1]) - (s[2] + s[3]);
      fre[2][h] = (c[0] - c[1]) + (c[2] - c[3]);  fim[2][h] = (s[0] - s[1]) + (s[2] - s[3]);
      fre[3][h] = (c[0] - c[1]) - (c[2] - c[3]);  fim[3][h] = (s[0] - s[1]) - (s[2] - s[3]);
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      split_pack2(fre[b][0], fre[b][1], oh[b][j2], ol[b][j2]);
      split_pack2(fim[b][0], fim[b][1], oh[b][8 + j2], ol[b][8 + j2]);
    }
  }
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const size_t o = ((size_t)(env * 4 + b) * SH_HP + x) * SH_K + kb * KB;     // halves
    st_global_v8(e_hi + o, oh[b]);
    st_global_v8(e_hi + o + 16, oh[b] + 8);
    st_global_v8(e_lo + o, ol[b]);
    st_global_v8(e_lo + o + 16, ol[b] + 8);
  }
}

// ----------------------------------------------------------------------------- camera, centroids, integrator
// Philox-4x32-10 (Salmon et al. 2011), one counter block per call.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c.x), l0 = 0xD2511F53u * c.x;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c.z), l1 = 0xCD9E8D57u * c.z;
    c = make_uint4(h1 ^ c.y ^ k.x, l1, h0 ^ c.w ^ k.y, l0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
__device__ __forceinline__ float u01(uint32_t r) { return ((float)(r >> 8) + 0.5f) * (1.0f / 16777216.0f); }   // (0, 1]: the top words round to 1 - 2^-23 and 1.0

// Photon count at rate lam (hcipy large_poisson, AO_env.py:274) in FP32 arithmetic:
//   lam > 1e6      rounded normal, as large_poisson itself does
//   lam >= 10      normal quantile with the Cornish-Fisher skewness and kurtosis terms of the Poisson law
//                  (k = lam + sqrt(lam) z + (z^2 - 1) / 6 - (z^3 - z) / (72 sqrt(lam)), rounded): mean, variance and
//                  third moment of Poisson(lam) to O(1 / lam) -- the camera's pixels sit at 1e1 ... 1e7 photons
//   lam < 10       Knuth's product of uniforms (exact)
// The common branch takes one standard normal z (the caller makes four of them, for the four mirror pixels, from ONE
// Philox block by two Box-Muller transforms); the rare small-rate branch draws its own blocks at ctr.w = 1 + 4 n + m.
__device__ __forceinline__ float sqrt_fast(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __noinline__ float poisson_small_f32(float lam, uint4 ctr, uint2 key, int m) {
  if (!(lam > 0.f)) return 0.f;
  const float enlam = __expf(-lam);
  float prod = 1.f;
  int k = 0;
  for (uint32_t nblk = 0;; ++nblk) {
    uint4 c2 = ctr;
    c2.w = 1u + 4u * nblk + (uint32_t)m;
    const uint4 blk = philox4x32_10(c2, key);
    const uint32_t w[4] = {blk.x, blk.y, blk.z, blk.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      prod *= u01(w[j]);
      if (prod > enlam) ++k; else return (float)k;
    }
  }
}
__device__ __forceinline__ float poisson_large_f32(float lam, float z) {
  // rounding to an integer adds 1/12 of variance: taken off the normal's scale, so that var = lam
  const float sl = sqrt_fast(lam - (1.f / 12.f));
  const float z2 = z * z;
  // above 1e6 the correction terms are below the rounding of lam itself: large_poisson's plain rounded normal
  const float corr = lam > 1e6f ? 0.f : (z2 - 1.f) * (1.f / 6.f) - (z2 * z - z) * __fdividef(1.f, 72.f * sl);
  return fmaxf(rintf(fmaf(sl, z, lam) + corr), 0.f);
}
// four standard normals from one counter block
__device__ __forceinline__ void normals4(uint4 r, float* z) {
  const float ra = sqrt_fast(-2.f * __logf(u01(r.x))), rb = sqrt_fast(-2.f * __logf(u01(r.z)));
  float s, c;
  __sincosf(6.28318530718f * u01(r.y), &s, &c);
  z[0] = ra * c; z[1] = ra * s;
  __sincosf(6.28318530718f * u01(r.w), &s, &c);
  z[2] = rb * c; z[3] = rb * s;
}

struct ShCamParams {
  const float* G;            // [env][p][q][128 i'][re 128 | im 128]
  const int16_t* slot;       // [P] selected-lenslet slot of each camera pixel, -1 = none
  const double* slotc;       // [Nsub][3] pixels, sum of columns, sum of rows of each slot (the + 1e-10 term, AO_env.py:277)
  const double* offset;      // [2][Nsub]
  const double* recon;       // [K][2 Nsub]
  double* act_sh;            // [B][K]
  double* action_out;        // [B][K] or null
  int Nsub, K, env0, noise_mode, qshift;
  float img_scale;           // amp^2 x pixel area x dt / table scales
  double X0, dX, Y0, dY;     // detector coordinates: x = X0 + dX col, y = Y0 + dY row
  unsigned long long seed, env_id_base, draw;
};

// Block per environment, thread = (fold column u, one of CAM_PARTS row ranges): walks its fold rows, reads the four
// blocks (coalesced along u), unfolds to the four mirror pixels, image = |F|^2 x scale, photon noise (one Philox
// block per fold pixel), and adds every pixel to its lenslet's (flux, flux x col, flux x row) sums.  A thread keeps
// the running sums of its four pixel streams in registers (FP64, fixed order) and, when the lenslet changes (every 20
// rows), adds them to the block's sums in 64-bit FIXED POINT through shared-memory atomics: integer addition does
// not depend on the order of the additions, so the result is deterministic like the FP64 path's per-lenslet warps.
constexpr int CAM_PARTS = 2, CAM_THREADS = 128 * CAM_PARTS;
__global__ void __launch_bounds__(CAM_THREADS, 2) k_sh_camera_tc(const ShCamParams p) {
  constexpr int Np = TC_NP;
  extern __shared__ unsigned long long cam_acc[];       // [3 Nsub] fixed-point sums, then [2 Nsub] doubles (slopes)
  double* slopes = reinterpret_cast<double*>(cam_acc + 3 * p.Nsub);
  const int b = blockIdx.x, u = threadIdx.x & 127, part = threadIdx.x >> 7;
  for (int i = threadIdx.x; i < 3 * p.Nsub; i += blockDim.x) cam_acc[i] = 0ull;
  __syncthreads();
  {
    const bool active = u < SH_NH;
    const int uu = active ? u : 0;
    const int lane = threadIdx.x & 31;
    const float* g = p.G + (size_t)b * 4 * SH_HP * (2 * SH_HP) + uu;
    const double qs = (double)(1ull << p.qshift);
    const unsigned long long genv = p.env_id_base + p.env0 + b;
    const uint2 key = make_uint2((uint32_t)p.seed ^ (uint32_t)(genv >> 32), (uint32_t)(p.seed >> 32) ^ (uint32_t)(p.draw >> 32));
    const bool noisy = p.noise_mode == AOG_SH_NOISE_POISSON;
    int cur[4] = {-1, -1, -1, -1};
    double f[4] = {0, 0, 0, 0}, sy[4] = {0, 0, 0, 0};
    // Warp-collective flush of stream m for the lanes with `need`: the lanes of a warp that sit in the same lenslet
    // are neighbours, so a segmented scan over equal slots leaves each lenslet's total in its last lane, which alone
    // touches shared memory (<= 3 atomics per warp and sum instead of 32 colliding ones).
    auto flush = [&](int m, bool need) {
      const bool give = need && cur[m] >= 0 && f[m] != 0.0;
      const int k = give ? cur[m] : -1 - lane;                       // distinct negative keys: never merged
      const int col = (m & 2) ? Np - 1 - uu : uu;
      long long a = give ? __double2ll_rn(f[m] * qs) : 0ll;
      long long bx = a * col;                                        // the column is fixed along a stream
      long long cy = give ? __double2ll_rn(sy[m] * qs) : 0ll;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int ko = __shfl_up_sync(0xffffffffu, k, o);
        const long long ao = __shfl_up_sync(0xffffffffu, a, o), bo = __shfl_up_sync(0xffffffffu, bx, o),
                        co = __shfl_up_sync(0xffffffffu, cy, o);
        if (lane >= o && ko == k) { a += ao; bx += bo; cy += co; }
      }
      const int kn = __shfl_down_sync(0xffffffffu, k, 1);
      if (give && (lane == 31 || kn != k)) {
        atomicAdd(&cam_acc[3 * k], (unsigned long long)a);
        atomicAdd(&cam_acc[3 * k + 1], (unsigned long long)bx);
        atomicAdd(&cam_acc[3 * k + 2], (unsigned long long)cy);
      }
      if (need) f[m] = sy[m] = 0.0;
    };
    constexpr int ROWS = SH_NH / CAM_PARTS;
    float nre[4], nim[4];                 // the next row's blocks, loaded one row ahead of the arithmetic
    int nsl[4];
    auto fetch = [&](int i) {
#pragma unroll
      for (int blk = 0; blk < 4; ++blk) {
        const float* r = g + ((size_t)blk * SH_HP + i) * (2 * SH_HP);
        nre[blk] = __ldg(r);
        nim[blk] = __ldg(r + SH_HP);
      }
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int row = (m & 1) ? Np - 1 - i : i, col = (m & 2) ? Np - 1 - uu : uu;
        nsl[m] = active ? (int)__ldg(p.slot + row * Np + col) : -1;
      }
    };
    fetch(part * ROWS);
    for (int i = part * ROWS; i < (part + 1) * ROWS; ++i) {
      float re[4], im[4];
      int slv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { re[k] = nre[k]; im[k] = nim[k]; slv[k] = nsl[k]; }
      if (i + 1 < (part + 1) * ROWS) fetch(i + 1);
      // blocks: 0 = (p+, q+), 1 = (p+, q-), 2 = (p-, q+), 3 = (p-, q-);  p = row fold, q = column fold
      // pixel m: 0 = (i, u), 1 = (N-1-i, u), 2 = (i, N-1-u), 3 = (N-1-i, N-1-u)
      const float fr[4] = {(re[0] + re[1]) + (re[2] + re[3]), (re[0] + re[1]) - (re[2] + re[3]),
                           (re[0] - re[1]) + (re[2] - re[3]), (re[0] - re[1]) - (re[2] - re[3])};
      const float fi[4] = {(im[0] + im[1]) + (im[2] + im[3]), (im[0] + im[1]) - (im[2] + im[3]),
                           (im[0] - im[1]) + (im[2] - im[3]), (im[0] - im[1]) - (im[2] - im[3])};
      float v[4];
      bool small = false;
#pragma unroll
      for (int m = 0; m < 4; ++m) v[m] = slv[m] >= 0 ? (fr[m] * fr[m] + fi[m] * fi[m]) * p.img_scale : 0.f;
      // lenslet rows end together: one vote per row, and normally the whole warp flushes at once
      const bool changed = slv[0] != cur[0] || slv[1] != cur[1] || slv[2] != cur[2] || slv[3] != cur[3];
      if (__any_sync(0xffffffffu, changed)) {
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const bool need = slv[m] != cur[m];
          flush(m, need);
          cur[m] = slv[m];
        }
      }
      // rows / warps that only see unselected lenslets (the aperture's rim and corners) have nothing to add
      if (!__any_sync(0xffffffffu, slv[0] >= 0 || slv[1] >= 0 || slv[2] >= 0 || slv[3] >= 0)) continue;
      if (noisy) {
        const uint4 ctr = make_uint4((uint32_t)(i * SH_NH + uu), (uint32_t)genv, (uint32_t)p.draw, 0u);
        float z[4];
        normals4(philox4x32_10(ctr, key), z);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          small |= v[m] > 0.f && v[m] < 10.f;
          v[m] = v[m] > 0.f ? poisson_large_f32(fmaxf(v[m], 10.f), z[m]) : 0.f;      // (rates below 10 are redone exactly below)
        }
        if (__any_sync(0xffffffffu, small)) {                        // rare: a pixel with fewer than 10 photons
#pragma unroll 1
          for (int m = 0; m < 4; ++m) {
            const float lam = slv[m] >= 0 ? (fr[m] * fr[m] + fi[m] * fi[m]) * p.img_scale : 0.f;
            if (lam > 0.f && lam < 10.f) {
              const float k = poisson_small_f32(lam, ctr, key, m);
              if (m == 0) v[0] = k; else if (m == 1) v[1] = k; else if (m == 2) v[2] = k; else v[3] = k;
            }
          }
        }
      }
      const double r0 = (double)i, r1 = (double)(Np - 1 - i);
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        f[m] += (double)v[m];
        sy[m] = fma((double)v[m], (m & 1) ? r1 : r0, sy[m]);
      }
    }
#pragma unroll
    for (int m = 0; m < 4; ++m) flush(m, true);
  }
  __syncthreads();
  const double inv_q = 1.0 / (double)(1ull << p.qshift);
  for (int m = threadIdx.x; m < p.Nsub; m += blockDim.x) {
    const double fl = (double)(long long)cam_acc[3 * m] * inv_q + 1e-10 * p.slotc[3 * m];
    const double cx = ((double)(long long)cam_acc[3 * m + 1] * inv_q + 1e-10 * p.slotc[3 * m + 1]) / fl;
    const double cy = ((double)(long long)cam_acc[3 * m + 2] * inv_q + 1e-10 * p.slotc[3 * m + 2]) / fl;
    slopes[m] = (p.X0 + p.dX * cx) - p.offset[m];
    slopes[p.Nsub + m] = (p.Y0 + p.dY * cy) - p.offset[p.Nsub + m];
  }
  __syncthreads();
  // a <- 0.99 a - 0.3 R slopes (AO_env.py:282-285): one warp per reconstructor row, fixed-order tree sum
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int k = warp; k < p.K; k += nw) {
    double r = 0.0;
    for (int m = lane; m < 2 * p.Nsub; m += 32) r += p.recon[(size_t)k * 2 * p.Nsub + m] * slopes[m];
    r = warp_sum(r);
    if (lane == 0) {
      const size_t idx = (size_t)(p.env0 + b) * p.K + k;
      const double a = (1.0 - 0.01) * p.act_sh[idx] - 0.3 * r;
      p.act_sh[idx] = a;
      if (p.action_out) p.action_out[idx] = a;
    }
  }
}

// test hook (aog_debug_poisson, FP32 sampler): draw i at rate lam from counter block i
__global__ void k_debug_poisson_f32(float lam, int n, unsigned long long seed, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const uint4 ctr = make_uint4((uint32_t)(i >> 2), 0x51u, 0u, 0u);
  float z[4];
  normals4(philox4x32_10(ctr, key), z);
  out[i] = (double)(lam >= 10.f ? poisson_large_f32(lam, z[i & 3]) : poisson_small_f32(lam, ctr, key, i & 3));
}

// test hook (aog_debug_normals): block i -> raw[i] = Philox-4x32-10 of (counter words[6 i .. 6 i + 3], key
// words[6 i + 4 .. 6 i + 5]) when `philox`, else raw[i] = words[4 i .. 4 i + 3]; z[4 i ..] = the four normals of raw[i]
// by the extrusion / synthesis generator (cam = 0: aog_philox4x32_10, aog_normals4) or the camera's (cam = 1)
__global__ void k_debug_normals(const uint32_t* __restrict__ words, int n, int philox, int cam,
                                uint32_t* __restrict__ raw, float* __restrict__ z) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint4 r;
  if (philox) {
    const uint32_t* w = words + (size_t)6 * i;
    const uint4 c = make_uint4(w[0], w[1], w[2], w[3]);
    const uint2 k = make_uint2(w[4], w[5]);
    r = cam ? philox4x32_10(c, k) : aog_philox4x32_10(c, k);
    raw[4 * (size_t)i] = r.x; raw[4 * (size_t)i + 1] = r.y; raw[4 * (size_t)i + 2] = r.z; raw[4 * (size_t)i + 3] = r.w;
  } else {
    const uint32_t* w = words + (size_t)4 * i;
    r = make_uint4(w[0], w[1], w[2], w[3]);
  }
  float o[4];
  if (cam) normals4(r, o); else aog_normals4(r, o);
#pragma unroll
  for (int k = 0; k < 4; ++k) z[4 * (size_t)i + k] = o[k];
}

// ----------------------------------------------------------------------------- host side
// Operator table of one stage: C' = C diag(exp(i g)) (micro-lens phase folded in), checked for centrosymmetry,
// folded by parity (Ce/o[i'][i] = (C'[i'][i] +- C'[i'][N-1-i]) / 2), scaled by a power of two into the fp16 range,
// embedded in real arithmetic (rows re: [Cr | -Ci], rows im: [Ci | Cr] over K = 8 blocks of [16 re | 16 im]) and
// split hi + lo.  Layout [parity][re | im][128 rows][256 K]; padding rows / columns are zero.
int build_sh_operator(aog_env* env, TensorState* ts, int stage, const std::vector<double>& g) {
  const int N = TC_NP, H = SH_NH;
  const std::vector<double>& C = ts->h_shC;                // [N][N] complex
  std::vector<double> cr((size_t)N * N), ci((size_t)N * N);
  double mx = 0.0;
  for (int r = 0; r < N; ++r)
    for (int k = 0; k < N; ++k) {
      const double a = C[2 * ((size_t)r * N + k)], b = C[2 * ((size_t)r * N + k) + 1];
      const double cg = std::cos(g[k]), sg = std::sin(g[k]);
      cr[(size_t)r * N + k] = a * cg - b * sg;
      ci[(size_t)r * N + k] = a * sg + b * cg;
      mx = std::max(mx, std::max(std::fabs(a), std::fabs(b)));
    }
  double res = 0.0;
  for (int r = 0; r < N; ++r)
    for (int k = 0; k < N; ++k) {
      res = std::max(res, std::fabs(cr[(size_t)r * N + k] - cr[(size_t)(N - 1 - r) * N + (N - 1 - k)]));
      res = std::max(res, std::fabs(ci[(size_t)r * N + k] - ci[(size_t)(N - 1 - r) * N + (N - 1 - k)]));
    }
  if (!(res <= 1e-12 * mx)) { ts->sh_why = "Fresnel operator x micro-lens phase is not centrosymmetric"; return AOG_ERR_UNSUPPORTED; }
  double fmx = 0.0;
  std::vector<double> f[2][2];                             // [parity][re | im][H * H]
  for (int par = 0; par < 2; ++par)
    for (int c = 0; c < 2; ++c) f[par][c].assign((size_t)H * H, 0.0);
  for (int r = 0; r < H; ++r)
    for (int k = 0; k < H; ++k) {
      const double ar = cr[(size_t)r * N + k], br = cr[(size_t)r * N + (N - 1 - k)];
      const double ai = ci[(size_t)r * N + k], bi = ci[(size_t)r * N + (N - 1 - k)];
      f[0][0][(size_t)r * H + k] = 0.5 * (ar + br); f[0][1][(size_t)r * H + k] = 0.5 * (ai + bi);
      f[1][0][(size_t)r * H + k] = 0.5 * (ar - br); f[1][1][(size_t)r * H + k] = 0.5 * (ai - bi);
      for (int par = 0; par < 2; ++par)
        for (int c = 0; c < 2; ++c) fmx = std::max(fmx, std::fabs(f[par][c][(size_t)r * H + k]));
    }
  if (fmx == 0.0) { ts->sh_why = "Fresnel operator is zero"; return AOG_ERR_UNSUPPORTED; }
  int e = 0;
  std::frexp(fmx, &e);                                     // fmx = m 2^e, m in [0.5, 1)
  const double scale = std::ldexp(1.0, 5 - e);             // largest entry in [16, 32)
  ts->shScale[stage] = scale;
  std::vector<double> t((size_t)4 * SH_HP * SH_K, 0.0);
  for (int par = 0; par < 2; ++par)
    for (int r = 0; r < H; ++r)
      for (int k = 0; k < H; ++k) {
        const double re = f[par][0][(size_t)r * H + k] * scale, im = f[par][1][(size_t)r * H + k] * scale;
        const int kr = (k >> 4) * KB + (k & 15), ki = kr + 16;
        double* row_re = &t[((size_t)(par * 2 + 0) * SH_HP + r) * SH_K];
        double* row_im = &t[((size_t)(par * 2 + 1) * SH_HP + r) * SH_K];
        row_re[kr] = re;  row_re[ki] = -im;
        row_im[kr] = im;  row_im[ki] = re;
      }
  int rc;
  if ((rc = ts->shCE_hi[stage].alloc(env, t.size()))) return rc;
  if ((rc = ts->shCE_lo[stage].alloc(env, t.size()))) return rc;
  if ((rc = upload_split(env, t, ts->shCE_hi[stage], ts->shCE_lo[stage]))) return rc;
  if ((rc = make_map(env, &ts->tmShCE_hi[stage], ts->shCE_hi[stage], 4 * SH_HP, SH_HP, SH_K, KB))) return rc;
  if ((rc = make_map(env, &ts->tmShCE_lo[stage], ts->shCE_lo[stage], 4 * SH_HP, SH_HP, SH_K, KB))) return rc;
  return AOG_OK;
}

// All six SH tables are in: check the structure the kernels rely on and build the device operands.
int build_sh_tensor_tables(aog_env* env, TensorState* ts) {
  const int N = TC_NP, P = N * N, Nsub = env->sh_num_sub, npix = env->sh_num_pix;
  ts->sh_ready = false;
  ts->sh_unsupported = true;
  if (getenv("AOG_SH_F64") != nullptr) { ts->sh_why = "AOG_SH_F64 set"; return AOG_OK; }
  // micro-lens phase separable?  mla[y][x] = gy[y] + gx[x]
  const std::vector<double>& mla = ts->h_shMla;
  std::vector<double> gy(N), gx(N);
  for (int y = 0; y < N; ++y) gy[y] = mla[(size_t)y * N] - 0.5 * mla[0];
  for (int x = 0; x < N; ++x) gx[x] = mla[x] - 0.5 * mla[0];
  double res = 0.0;
  for (int y = 0; y < N; ++y)
    for (int x = 0; x < N; ++x) res = std::max(res, std::fabs(mla[(size_t)y * N + x] - gy[y] - gx[x]));
  if (!(res <= 1e-9)) { ts->sh_why = "micro-lens phase is not separable"; return AOG_OK; }
  int rc = build_sh_operator(env, ts, 0, gy);              // first product contracts the rows y
  if (rc == AOG_ERR_UNSUPPORTED) return AOG_OK;
  if (rc) return rc;
  rc = build_sh_operator(env, ts, 1, gx);                  // second product contracts the columns x
  if (rc == AOG_ERR_UNSUPPORTED) return AOG_OK;
  if (rc) return rc;
  // camera pixels -> lenslet slots; detector coordinates affine in (col, row)
  std::vector<int16_t> slot((size_t)P, (int16_t)-1);
  std::vector<double> slotc((size_t)3 * Nsub, 0.0);
  if (Nsub > 32767) { ts->sh_why = "too many lenslets"; return AOG_OK; }
  for (int m = 0; m < Nsub; ++m)
    for (int i = ts->h_shOff[m]; i < ts->h_shOff[m + 1]; ++i) {
      const int pix = ts->h_shPix[i];
      if (pix < 0 || pix >= P || slot[pix] != -1) { ts->sh_why = "lenslet pixel lists overlap"; return AOG_OK; }
      slot[pix] = (int16_t)m;
      slotc[3 * m] += 1.0;
      slotc[3 * m + 1] += (double)(pix % N);
      slotc[3 * m + 2] += (double)(pix / N);
    }
  // x = X0 + dX col, y = Y0 + dY row: least squares is overkill -- two reference pixels, then verify all
  double X0 = 0, dX = 0, Y0 = 0, dY = 0;
  {
    int i0 = -1, ic = -1, ir = -1;
    for (int i = 0; i < npix && (ic < 0 || ir < 0); ++i) {
      if (i0 < 0) { i0 = i; continue; }
      if (ic < 0 && ts->h_shPix[i] % N != ts->h_shPix[i0] % N) ic = i;
      if (ir < 0 && ts->h_shPix[i] / N != ts->h_shPix[i0] / N) ir = i;
    }
    if (i0 < 0 || ic < 0 || ir < 0) { ts->sh_why = "degenerate lenslet pixel list"; return AOG_OK; }
    const int c0 = ts->h_shPix[i0] % N, r0 = ts->h_shPix[i0] / N;
    dX = (ts->h_shPx[ic] - ts->h_shPx[i0]) / (double)(ts->h_shPix[ic] % N - c0);
    dY = (ts->h_shPy[ir] - ts->h_shPy[i0]) / (double)(ts->h_shPix[ir] / N - r0);
    X0 = ts->h_shPx[i0] - dX * c0;
    Y0 = ts->h_shPy[i0] - dY * r0;
    const double tol = 1e-9 * (std::fabs(dX) + std::fabs(dY)) * N;
    for (int i = 0; i < npix; ++i) {
      const int c = ts->h_shPix[i] % N, r = ts->h_shPix[i] / N;
      if (std::fabs(X0 + dX * c - ts->h_shPx[i]) > tol || std::fabs(Y0 + dY * r - ts->h_shPy[i]) > tol) {
        ts->sh_why = "detector coordinates are not a uniform separable grid";
        return AOG_OK;
      }
    }
  }
  ts->shX0 = X0; ts->shdX = dX; ts->shY0 = Y0; ts->shdY = dY;
  if ((rc = ts->shSlot.alloc(env, slot.size()))) return rc;
  if ((rc = ts->shSlotC.alloc(env, slotc.size()))) return rc;
  AOG_CUDA(cudaMemcpy(ts->shSlot, slot.data(), slot.size() * sizeof(int16_t), cudaMemcpyHostToDevice));
  AOG_CUDA(cudaMemcpy(ts->shSlotC, slotc.data(), slotc.size() * sizeof(double), cudaMemcpyHostToDevice));
  ts->sh_unsupported = false;
  ts->sh_ready = true;
  ts->sh_why.clear();
  return AOG_OK;
}

int ensure_sh_tensor_buffers(aog_env* env, TensorState* ts) {
  if (ts->sh_buffers) return AOG_OK;
  const size_t ch = env->chunk, P = env->P;
  const size_t rows = ch * 4 * SH_HP, nel = rows * SH_K;
  int rc;
  if (!ts->phi) {
    if ((rc = ts->phi.alloc(env, ch * P))) return rc;
    AOG_CUDA(cudaMemset(ts->phi, 0, ch * P * sizeof(float)));
  }
  if ((rc = ts->shEB_hi.alloc(env, nel))) return rc;
  if ((rc = ts->shEB_lo.alloc(env, nel))) return rc;
  if ((rc = ts->shYB_hi.alloc(env, nel))) return rc;
  if ((rc = ts->shYB_lo.alloc(env, nel))) return rc;
  if ((rc = ts->shG.alloc(env, nel))) return rc;
  // padding rows / columns of the operands are never written: they must be zero (and finite)
  AOG_CUDA(cudaMemset(ts->shEB_hi, 0, nel * sizeof(__half)));
  AOG_CUDA(cudaMemset(ts->shEB_lo, 0, nel * sizeof(__half)));
  AOG_CUDA(cudaMemset(ts->shYB_hi, 0, nel * sizeof(__half)));
  AOG_CUDA(cudaMemset(ts->shYB_lo, 0, nel * sizeof(__half)));
  AOG_CUDA(cudaMemset(ts->shG, 0, nel * sizeof(float)));
  if ((rc = make_map(env, &ts->tmShEB_hi, ts->shEB_hi, rows, SH_HP, SH_K, KB))) return rc;
  if ((rc = make_map(env, &ts->tmShEB_lo, ts->shEB_lo, rows, SH_HP, SH_K, KB))) return rc;
  if ((rc = make_map(env, &ts->tmShYB_hi, ts->shYB_hi, rows, SH_HP, SH_K, KB))) return rc;
  if ((rc = make_map(env, &ts->tmShYB_lo, ts->shYB_lo, rows, SH_HP, SH_K, KB))) return rc;
  if ((rc = make_map(env, &ts->tmShYout_hi, ts->shYB_hi, rows, SH_HP, SH_K, 16))) return rc;
  if ((rc = make_map(env, &ts->tmShYout_lo, ts->shYB_lo, rows, SH_HP, SH_K, 16))) return rc;
  AOG_CUDA(cudaFuncSetAttribute(k_sh_gemm<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SG_SMEM_BYTES));
  AOG_CUDA(cudaFuncSetAttribute(k_sh_gemm<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SG_SMEM_BYTES));
  ts->sh_buffers = true;
  return AOG_OK;
}

// phase -> folded field -> the two products for envs [e0, e0 + nB): leaves G in ts->shG
int sh_tensor_optics(aog_env* env, TensorState* ts, int e0, int nB, cudaStream_t st) {
  const aog_config& c = env->cfg;
  const int Np = TC_NP, K = c.num_modes;
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[2].get(), st));
  {   // the SH mirror's actuators -> half-turns of DM phase per unit mode, split fp16 (the DM GEMM's A operand)
    const int rows = cdiv(nB, 128) * 128;
    k_act_pack<<<cdiv(rows * ts->kpad, 256), 256, 0, st>>>(env->act_sh, ts->act_hi, ts->act_lo, K, ts->kpad, e0, nB, rows,
                                                           4.0 / c.wavelength_wfs);
    AOG_LAUNCH_CHECK();
    ts->packed_valid = false;
    FieldParams fp{};
    fp.num_envs = nB;
    fp.num_items = cdiv(nB, 128) * Np;
    fp.items_per_cta = std::max(FK_MIN_ITEMS, cdiv(fp.num_items, ts->num_sms));
    fp.nkb = ts->kpad / 64;
    fp.col_origin = (int)env->cnt.column_origin;
    fp.env0 = e0;
    fp.dbg = 0;
    fp.sci_ratio_q32 = 0;
    fp.apmask = ts->apmask; fp.m1o32 = ts->m1o32; fp.phi = ts->phi; fp.R4 = ts->R4;
    fp.strehl_part = env->strehl_part; fp.gfib = nullptr; fp.fib_part = nullptr; fp.err_flag = ts->err_flag;
    int rc = launch_phase<false, 1, 3>(env, ts, fp, cdiv(fp.num_items, fp.items_per_cta), st);
    if (rc) return rc;
    // nothing after this kernel reads the screens or the phase tiles: the next aog_step may extrude concurrently
    // (single-chunk handles; see aog_step)
    if (nB == c.num_envs) {
      AOG_CUDA(cudaEventRecord(env->ev_sh_phase.get(), st));
      env->sh_phase_pending = true;
      env->sh_phase_stream = st;
    }
  }
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[3].get(), st));
  // k_sh_fold materialises the folded field and the first product streams it by TMA (forming it on chip inside the
  // first product was measured slower: DESIGN.md 4.4)
  k_sh_fold<<<dim3(SH_NKB, nB), 128, 0, st>>>(ts->phi, ts->apmask, ts->shEB_hi, ts->shEB_lo, nB);
  AOG_LAUNCH_CHECK();
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[4].get(), st));
  ShGemmParams gp{};
  gp.num_envs = nB;
  gp.G = ts->shG;
  { const char* d = getenv("AOG_SH_DEBUG"); gp.dbg = d ? atoi(d) : 0; }
  gp.err_flag = ts->err_flag;
  // clusters come in pairs (one per parity); each takes every (clusters / 2)-th environment
  const int clusters = std::max(2, std::min((ts->num_sms / 2) & ~1, 2 * nB));
  k_sh_gemm<1><<<2 * clusters, SG_THREADS, SG_SMEM_BYTES, st>>>(ts->tmShCE_hi[0], ts->tmShCE_lo[0], ts->tmShEB_hi, ts->tmShEB_lo,
                                                                ts->tmShYout_hi, ts->tmShYout_lo, gp);
  AOG_LAUNCH_CHECK();
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[5].get(), st));
  k_sh_gemm<2><<<2 * clusters, SG_THREADS, SG_SMEM_BYTES, st>>>(ts->tmShCE_hi[1], ts->tmShCE_lo[1], ts->tmShYB_hi, ts->tmShYB_lo,
                                                         ts->tmShYout_hi, ts->tmShYout_lo, gp);
  AOG_LAUNCH_CHECK();
  if (env->timing) AOG_CUDA(cudaEventRecord(env->tev[6].get(), st));
  return AOG_OK;
}

double sh_image_scale(const aog_env* env, const TensorState* ts) {
  const double s = ts->shScale[0] * ts->shScale[1];
  return env->sh_amplitude * env->sh_amplitude * env->sh_weight_dt / (s * s);
}

}  // namespace

int aog_tensor_sh_table(aog_env* env, int which, const void* host) {
  TensorState* ts = env->tensor.get();
  if (!ts || env->cfg.num_pupil_pixels != TC_NP) return AOG_OK;
  const size_t P = env->P;
  const double* d = static_cast<const double*>(host);
  const int32_t* iv = static_cast<const int32_t*>(host);
  switch (which) {
    case AOG_TABLE_SH_FRESNEL: ts->h_shC.assign(d, d + 2 * P); ts->sh_have[0] = true; break;
    case AOG_TABLE_SH_MLA_PHASE: ts->h_shMla.assign(d, d + P); ts->sh_have[1] = true; break;
    case AOG_TABLE_SH_PIX_OFFSETS: ts->h_shOff.assign(iv, iv + env->sh_num_sub + 1); ts->sh_have[2] = true; break;
    case AOG_TABLE_SH_PIX_INDEX: ts->h_shPix.assign(iv, iv + env->sh_num_pix); ts->sh_have[3] = true; break;
    case AOG_TABLE_SH_PIX_X: ts->h_shPx.assign(d, d + env->sh_num_pix); ts->sh_have[4] = true; break;
    case AOG_TABLE_SH_PIX_Y: ts->h_shPy.assign(d, d + env->sh_num_pix); ts->sh_have[5] = true; break;
    default: return AOG_OK;                      // offsets / reconstructor / initial actuators: read from the handle
  }
  for (bool h : ts->sh_have)
    if (!h) return AOG_OK;
  return build_sh_tensor_tables(env, ts);
}

int aog_tensor_sh_step(aog_env* env, int noise_mode, double* action_out_dev, cudaStream_t st) {
  TensorState* ts = env->tensor.get();
  if (!ts || !ts->sh_ready || noise_mode == AOG_SH_NOISE_INJECTED) return AOG_ERR_UNSUPPORTED;
  if (!(ts->have_modes && ts->have_ap)) AOG_FAIL(AOG_ERR_STATE, "tensor path tables incomplete");
  const aog_config& c = env->cfg;
  int rc = ensure_sh_tensor_buffers(env, ts);
  if (rc) return rc;
  const int B = c.num_envs, Nsub = env->sh_num_sub;
  // fixed-point scale of the lenslet sums: even if one lenslet caught the whole frame, flux x 240 stays below 2^62
  const double frame = env->sh_amplitude * env->sh_amplitude * env->sh_weight_dt * (double)env->P * (double)TC_NP;
  int qshift = 22;
  while (qshift > 0 && frame * std::ldexp(1.0, qshift) > 4.0e18) --qshift;
  for (int e0 = 0; e0 < B; e0 += env->chunk) {
    const int nB = std::min(env->chunk, B - e0);
    if ((rc = sh_tensor_optics(env, ts, e0, nB, st))) return rc;
    ShCamParams cp{};
    cp.G = ts->shG; cp.slot = ts->shSlot; cp.slotc = ts->shSlotC; cp.offset = env->t_sh_offset; cp.recon = env->t_sh_recon;
    cp.act_sh = env->act_sh; cp.action_out = action_out_dev;
    cp.Nsub = Nsub; cp.K = c.num_modes; cp.env0 = e0; cp.noise_mode = noise_mode; cp.qshift = qshift;
    cp.img_scale = (float)sh_image_scale(env, ts);
    cp.X0 = ts->shX0; cp.dX = ts->shdX; cp.Y0 = ts->shY0; cp.dY = ts->shdY;
    cp.seed = c.seed ^ 0xD1B54A32D192ED03ull; cp.env_id_base = (unsigned long long)c.env_id_base;
    cp.draw = (unsigned long long)env->sh_draws;
    k_sh_camera_tc<<<nB, CAM_THREADS, (size_t)Nsub * (3 * sizeof(unsigned long long) + 2 * sizeof(double)), st>>>(cp);
    AOG_LAUNCH_CHECK();
    if (env->timing) { AOG_CUDA(cudaEventRecord(env->tev[7].get(), st)); env->tev_sh_valid = true; }
  }
  return AOG_OK;
}

int aog_tensor_sh_image(aog_env* env, int env_index, double* host_out, size_t count) {
  TensorState* ts = env->tensor.get();
  if (!ts || !ts->sh_ready) AOG_FAIL(AOG_ERR_UNSUPPORTED, "tensor-core Shack-Hartmann path not available: " + (ts ? ts->sh_why : std::string("no tensor state")));
  if (count != (size_t)env->P) AOG_FAIL(AOG_ERR_INVALID, "count");
  int rc = ensure_sh_tensor_buffers(env, ts);
  if (rc) return rc;
  cudaStream_t st = env->own_stream.get();
  // the phase kernel works on whole 128-env blocks of the tiled screens: run the block that holds env_index
  const int e0 = env_index & ~127, nB = std::min(128, env->cfg.num_envs - e0);
  if ((rc = sh_tensor_optics(env, ts, e0, nB, st))) return rc;
  const size_t nel = (size_t)4 * SH_HP * SH_K;
  std::vector<float> g(nel);
  AOG_CUDA(cudaMemcpyAsync(g.data(), ts->shG + (size_t)(env_index - e0) * nel, nel * sizeof(float), cudaMemcpyDeviceToHost, st));
  AOG_CUDA(cudaStreamSynchronize(st));
  const double sc = sh_image_scale(env, ts);
  const int N = TC_NP;
  for (int i = 0; i < SH_NH; ++i)
    for (int u = 0; u < SH_NH; ++u) {
      double re[4], im[4];
      for (int b = 0; b < 4; ++b) {
        re[b] = g[((size_t)b * SH_HP + i) * SH_K + u];
        im[b] = g[((size_t)b * SH_HP + i) * SH_K + SH_HP + u];
      }
      const double sgn[4][4] = {{1, 1, 1, 1}, {1, 1, -1, -1}, {1, -1, 1, -1}, {1, -1, -1, 1}};
      for (int m = 0; m < 4; ++m) {
        double fr = 0, fi = 0;
        for (int b = 0; b < 4; ++b) { fr += sgn[m][b] * re[b]; fi += sgn[m][b] * im[b]; }
        const int row = (m & 1) ? N - 1 - i : i, col = (m & 2) ? N - 1 - u : u;
        host_out[(size_t)row * N + col] = (fr * fr + fi * fi) * sc;
      }
    }
  return AOG_OK;
}

int aog_tensor_debug_poisson(int device, double lambda, int n, uint64_t seed, double* host_out) {
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return AOG_ERR_CUDA;
  DevArray<double> d;
  if (d.alloc(n) != cudaSuccess) return AOG_ERR_CUDA;
  k_debug_poisson_f32<<<cdiv(n, 256), 256>>>((float)lambda, n, (unsigned long long)seed, d);
  const cudaError_t e = cudaMemcpy(host_out, d, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? AOG_OK : AOG_ERR_CUDA;
}

int aog_tensor_debug_normals(int device, int generator, int philox, int n, const uint32_t* words_in, uint32_t* raw_out,
                             float* normals_out) {
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return AOG_ERR_CUDA;
  const size_t nw = (size_t)n * (philox ? 6 : 4), nr = philox ? (size_t)n * 4 : 0, nz = (size_t)n * 4;
  DevArray<uint32_t> d;                                           // [words | raw | normals]
  if (d.alloc(nw + nr + nz) != cudaSuccess) return AOG_ERR_CUDA;
  float* dz = reinterpret_cast<float*>(d + nw + nr);
  cudaError_t e = cudaMemcpy(d, words_in, nw * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_debug_normals<<<cdiv(n, 256), 256>>>(d, n, philox, generator, d + nw, dz);
    e = cudaMemcpy(normals_out, dz, nz * sizeof(float), cudaMemcpyDeviceToHost);
  }
  if (e == cudaSuccess && philox) e = cudaMemcpy(raw_out, d + nw, nr * sizeof(uint32_t), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? AOG_OK : AOG_ERR_CUDA;
}
