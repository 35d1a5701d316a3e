// Packed FP32x2 arithmetic for sm_100 (SASS FFMA2 / FADD2): one issue slot for two FP32 operations.  Each lane is the
// ordinary round-to-nearest FP32 operation (no flush to zero), so f2_fma(a, b, c).x == fmaf(a.x, b.x, c.x) bit for bit.
// The fused phase kernel uses them for the per-pixel steps it would otherwise issue once per pixel (phase rounding,
// angle scaling), two pixels at a time.  The float2 halves travel in a .b64 register pair; ptxas allocates them as one.
#pragma once

#define AOG_F32X2_OP(name, op)                                                                                           \
  __device__ __forceinline__ float2 name(float2 a, float2 b) {                                                         \
    float2 d;                                                                                                            \
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t" op                           \
        " rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"                                                                     \
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                               \
    return d;                                                                                                            \
  }
AOG_F32X2_OP(f2_add, "add.rn.f32x2")
AOG_F32X2_OP(f2_sub, "sub.rn.f32x2")
#undef AOG_F32X2_OP

// a * b + c per lane, one rounding
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
