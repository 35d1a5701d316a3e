// DM phase -> int32 fixed point (2^22 units per half-turn) without the conversion pipe.  The fused phase kernel rounds
// one TMEM accumulator per pixel; __float2int_rn is an F2I on the XU pipe, which the same pixel already loads with four
// MUFU sin / cos.  phase_fixed_rn issues two FP32 adds and two FMAs on the FMA pipe and one IMAD instead, and returns
// the same int32 as __float2int_rn(d * 2^22) for every |d| < 512 (|d * 2^22| < 2^31: every input the conversion does
// not saturate, which is also the whole range of the int32 phase).  tools/micro/phase_round_host.cu checks that
// exhaustively on the CPU (tests/test_phase_round.py).
#pragma once
#include <cstdint>
#include <cstring>

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
