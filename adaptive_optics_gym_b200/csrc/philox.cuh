// The generator of the extrusion noise and of the screen synthesis (kernels_f64.cuh), shared with the test hook
// aog_debug_normals (sh_tensor.cuh).
#pragma once
#include <stdint.h>

// Philox-4x32-10 (Salmon et al. 2011), one counter block per call
__device__ __forceinline__ uint4 aog_philox4x32_10(uint4 c, uint2 k) {
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
// four standard normals from one block: two Box-Muller transforms in FP32 on the SFU (24-bit uniforms in (0, 1]; over all
// of them within 3.5e-5 of an FP64 Box-Muller on B200, |z| <= 5.9: tests/test_device_noise_gpu.py).  The draws only
// have to be normal and reproducible from (seed, env, index) -- parity with the reference is through injected noise --
// and curand's FP64 Box-Muller cost 58 us per step of 4096 envs at 20 m/s.
__device__ __forceinline__ void aog_normals4(uint4 r, float (&z)[4]) {
  const float u0 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
  const float u2 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = ((float)(r.w >> 8) + 0.5f) * (1.0f / 16777216.0f);
  const float ra = sqrtf(-2.f * __logf(u0)), rb = sqrtf(-2.f * __logf(u2));
  float sn, cs;
  __sincosf(6.28318530718f * u1, &sn, &cs);
  z[0] = ra * cs; z[1] = ra * sn;
  __sincosf(6.28318530718f * u3, &sn, &cs);
  z[2] = rb * cs; z[3] = rb * sn;
}
