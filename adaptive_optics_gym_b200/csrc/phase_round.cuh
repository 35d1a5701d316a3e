// DM phase -> int32 fixed point (2^22 units per half-turn) without the conversion pipe.  The fused phase kernel rounds
// one TMEM accumulator per pixel; __float2int_rn is an F2I on the XU pipe, which the same pixel already loads with four
// MUFU sin / cos.  phase_fixed_rn issues two FP32 adds and two FMAs on the FMA pipe and one IMAD instead, and returns
// the same int32 as __float2int_rn(d * 2^22) for every |d| < 512 (|d * 2^22| < 2^31: every input the conversion does
// not saturate, which is also the whole range of the int32 phase).  tools/micro/phase_round_host.cu checks that
// exhaustively on the CPU (tests/test_phase_round.py).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#ifdef __CUDACC__
#include "fp32x2.cuh"
#endif

__host__ __device__ __forceinline__ uint32_t phase_round_bits(float f) {
#ifdef __CUDA_ARCH__
  return __float_as_uint(f);
#else
  uint32_t u;
  std::memcpy(&u, &f, sizeof u);
  return u;
#endif
}

// x = d 2^22 is exact (power-of-two scale).  x + 1.5 2^32 lands in [2^32, 2^33), where the FP32 spacing is 2^9: the sum
// is x rounded to a multiple of 2^9 (hi), and its bits count hi / 2^9 up from those of 1.5 2^32.  r = x - hi is exact
// with |r| <= 256, and r + 1.5 2^23 rounds it to an integer the same way.  hi is even, so rounding r to nearest, ties
// to even, rounds x to nearest, ties to even.
__host__ __device__ __forceinline__ int32_t phase_fixed_rn(float d) {
  const float x = d * 4194304.f;
  const float s = x + 6442450944.f;               // 1.5 * 2^32
  const float r = x - (s - 6442450944.f);
  const float u = r + 12582912.f;                 // 1.5 * 2^23
  return (int32_t)(((phase_round_bits(s) - 0x4FC00000u) << 9) + (phase_round_bits(u) - 0x4B400000u));
}

// Two pixels at once, the FP steps as packed FP32x2 operations (fp32x2.cuh) and the integer tail per pixel; returns
// phase_fixed_rn(d0), phase_fixed_rn(d1).  The scale folds into the FMAs: d 2^22 is exact, so fma(d, 2^22, c) rounds as
// x + c does, and fma(d, 2^22, -(s - 1.5 2^32)) is the exact r.  Four packed operations for two pixels instead of five
// scalar ones per pixel.  The host form runs the same steps per lane (tools/micro/phase_round_host.cu checks it).
__host__ __device__ __forceinline__ void phase_fixed_rn2(float d0, float d1, int32_t* r0, int32_t* r1) {
#ifdef __CUDA_ARCH__
  const float2 d = make_float2(d0, d1);
  const float2 s = f2_fma(d, make_float2(4194304.f, 4194304.f), make_float2(6442450944.f, 6442450944.f));
  const float2 nh = f2_sub(make_float2(6442450944.f, 6442450944.f), s);     // -hi
  const float2 u = f2_add(f2_fma(d, make_float2(4194304.f, 4194304.f), nh), make_float2(12582912.f, 12582912.f));
  const float s0 = s.x, s1 = s.y, u0 = u.x, u1 = u.y;
#else
  const float s0 = std::fma(d0, 4194304.f, 6442450944.f), s1 = std::fma(d1, 4194304.f, 6442450944.f);
  const float u0 = std::fma(d0, 4194304.f, 6442450944.f - s0) + 12582912.f;
  const float u1 = std::fma(d1, 4194304.f, 6442450944.f - s1) + 12582912.f;
#endif
  *r0 = (int32_t)(((phase_round_bits(s0) - 0x4FC00000u) << 9) + (phase_round_bits(u0) - 0x4B400000u));
  *r1 = (int32_t)(((phase_round_bits(s1) - 0x4FC00000u) << 9) + (phase_round_bits(u1) - 0x4B400000u));
}
