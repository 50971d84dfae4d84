// Device-side f32 vector math and the leaf helpers of src/common/math.rs / spectrum.rs.
// The whole library is compiled with -fmad=false, IEEE division and sqrt, no fast-math: every
// expression below evaluates in source order exactly like the reference's rustc/LLVM build, which is
// what makes primitive ids, t and barycentrics bit-identical to the CPU path.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#define PT_DEV __device__ __forceinline__
#define PT_DEVN static __device__ __noinline__

namespace ptrs {

struct V3 {
  float x, y, z;
};
PT_DEV V3 mk3(float x, float y, float z) { return V3{x, y, z}; }
PT_DEV V3 mk3(float4 v) { return V3{v.x, v.y, v.z}; }
PT_DEV V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
PT_DEV V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
PT_DEV V3 operator-(V3 a) { return {-a.x, -a.y, -a.z}; }
PT_DEV V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
PT_DEV V3 operator*(float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
PT_DEV V3 operator/(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
PT_DEV float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
PT_DEV V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
PT_DEV float norm_squared(V3 a) { return dot(a, a); }
PT_DEV float norm(V3 a) { return sqrtf(norm_squared(a)); }
PT_DEV V3 normalize(V3 a) {
  float n = norm(a);
  return {a.x / n, a.y / n, a.z / n};
}
PT_DEV V3 vabs(V3 a) { return {fabsf(a.x), fabsf(a.y), fabsf(a.z)}; }
PT_DEV float comp(V3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
PT_DEV void set_comp(V3& a, int i, float v) {
  if (i == 0) a.x = v;
  else if (i == 1) a.y = v;
  else a.z = v;
}
PT_DEV bool is_zero3(V3 a) { return a.x == 0.f && a.y == 0.f && a.z == 0.f; }

struct V2 {
  float x, y;
};

PT_DEV float rclamp(float v, float lo, float hi) { return v < lo ? lo : (v > hi ? hi : v); }  // f32::clamp

// src/common/math.rs ------------------------------------------------------------------------------
#define PT_MACHINE_EPSILON (1.1920929e-7f * 0.5f)
#define PT_ONE_MINUS_EPSILON 0x1.fffffep-1f
#define PT_PI 3.14159274f
#define PT_FRAC_1_PI 0.318309873f
#define PT_INV_2_PI (0.31830987f * 0.5f)
#define PT_FRAC_PI_2 1.57079637f
#define PT_FRAC_PI_4 0.785398185f
#define PT_HALF_MAX_I32 (2147483647 / 2)

PT_DEV float gamma_n(uint32_t n) { return ((float)n * PT_MACHINE_EPSILON) / (1.0f - (float)n * PT_MACHINE_EPSILON); }  // math.rs:8
PT_DEV int max_dimension(V3 v) {  // math.rs:12-26
  if (v.x > v.y) return v.x > v.z ? 0 : 2;
  return v.y > v.z ? 1 : 2;
}
PT_DEV V3 face_forward(V3 n, V3 v) { return dot(n, v) < 0.0f ? -n : n; }  // math.rs:37-46
PT_DEV void coordinate_system(V3 v1, V3* v2, V3* v3) {                    // math.rs:48-61
  if (fabsf(v1.x) > fabsf(v1.y)) *v2 = mk3(-v1.z, 0.0f, v1.x) / sqrtf(v1.x * v1.x + v1.z * v1.z);
  else *v2 = mk3(0.0f, v1.z, -v1.y) / sqrtf(v1.y * v1.y + v1.z * v1.z);
  *v3 = cross(v1, *v2);
}
// Written with selects instead of branches (three rays are offset per bounce, per component): same values.
PT_DEV float next_float_up(float v) {  // math.rs:71-88
  const float vv = v == 0.0f ? 0.0f : v;  // `if v == -0.0 { v = 0.0 }` (true for either zero)
  uint32_t ui = __float_as_uint(vv);
  ui += vv >= 0.0f ? 1u : 0xffffffffu;
  return v == CUDART_INF_F ? v : __uint_as_float(ui);
}
// math.rs:90-105 — reference quirk kept on purpose: increments are swapped w.r.t. pbrt, so the
// value moves UP for either sign and +-0 becomes NaN (0x7fffffff).
PT_DEV float next_float_down(float v) {
  const float vv = v == 0.0f ? -0.0f : v;
  uint32_t ui = __float_as_uint(vv);
  ui += vv > 0.0f ? 1u : 0xffffffffu;
  return v == -CUDART_INF_F ? v : __uint_as_float(ui);
}
// `off > 0 ? next_float_up(v) : (off < 0 ? next_float_down(v) : v)` (math.rs:123-129) as one select chain: for a
// finite non-zero v both functions add the same +-1 to the bit pattern (the quirk above), they differ only at
// +-0 and at the infinity each one keeps.  Bit-identical to the nested calls for every (v, off), NaNs included;
// no branch, so the six origin offsets of a bounce do not split the warp eighteen ways.
PT_DEV float nudge_along(float v, float off) {
  const bool is_up = off > 0.0f, is_dn = off < 0.0f, zero = v == 0.0f;
  const uint32_t base = zero ? (is_up ? 0u : 0x80000000u) : __float_as_uint(v);
  const uint32_t delta = (zero ? is_up : (v > 0.0f)) ? 1u : 0xffffffffu;
  const bool keep = (is_up && v == CUDART_INF_F) || (is_dn && v == -CUDART_INF_F) || !(is_up || is_dn);
  return keep ? v : __uint_as_float(base + delta);
}
PT_DEV V3 offset_ray_origin(V3 p, V3 p_error, V3 n, V3 w) {  // math.rs:107-131
  float d = dot(vabs(n), p_error);
  V3 offset = d * n;
  if (dot(w, n) < 0.0f) offset = -offset;
  V3 po = p + offset;
  po.x = nudge_along(po.x, offset.x);
  po.y = nudge_along(po.y, offset.y);
  po.z = nudge_along(po.z, offset.z);
  return po;
}
PT_DEV bool solve_linear_system_2x2(float a00, float a01, float a10, float a11, float b0, float b1, float* x0, float* x1) {  // math.rs:149-165
  float det = a00 * a11 - a01 * a10;
  if (fabsf(det) < 1e-10f) return false;
  float r0 = (a11 * b0 - a01 * b1) / det;
  float r1 = (a00 * b1 - a10 * b0) / det;
  if (r0 != r0 || r1 != r1) return false;
  *x0 = r0;
  *x1 = r1;
  return true;
}
PT_DEV float power_heuristic(float f_pdf, float g_pdf) {  // math.rs:167-171 with nf = ng = 1
  float f = 1.0f * f_pdf, g = 1.0f * g_pdf;
  return (f * f) / (f * f + g * g);
}
PT_DEV float spherical_theta(V3 v) { return acosf(rclamp(v.z, -1.0f, 1.0f)); }  // math.rs:173
PT_DEV float spherical_phi(V3 v) {                                            // math.rs:177
  float p = atan2f(v.y, v.x);
  return p < 0.0f ? p + 2.0f * PT_PI : p;
}
PT_DEV int abs_mod(int a, int b) {  // math.rs:237-244
  int r = a - (a / b) * b;
  return r < 0 ? r + b : r;
}
// sinf / cosf of an angle below 105615 radians in magnitude, the range on which libdevice reduces the argument with three
// multiply-adds: its large-argument branch (Payne-Hanek, with a 28-byte local array) is compiled out, so the shade
// kernels that call these keep no local-memory frame.  Same values as sinf / cosf on that range, NaN included.
// PRECONDITION: |x| < 105615 or x is NaN.  A larger or infinite argument is undefined behaviour, not a wrong value; use
// sinf / cosf for any angle that is not bounded by construction.  The callers (concentric disk, GGX phi, environment
// sample, acos-based theta) all pass angles within [-2 pi, 2 pi]: a Sobol or table sample in [0, 1] scaled by at most
// 2 pi, or an acos.
PT_DEV float sin_small_angle(float x) {
  if (fabsf(x) >= 105615.0f) __builtin_unreachable();
  return sinf(x);
}
PT_DEV float cos_small_angle(float x) {
  if (fabsf(x) >= 105615.0f) __builtin_unreachable();
  return cosf(x);
}
PT_DEV float lerpf(float x, float y, float a) { return x * (1.0f - a) + y * a; }  // math.rs:250
PT_DEV uint64_t cantor_pairing(uint64_t x, uint64_t y) { return (x + y) * (x + y + 1) / 2 + y; }  // math.rs:256

// RGBSpectrum, src/common/spectrum.rs ----------------------------------------------------------------
struct Spec {
  float r, g, b;
};
PT_DEV Spec sp(float c) { return {c, c, c}; }
PT_DEV Spec sp(float r, float g, float b) { return {r, g, b}; }
PT_DEV Spec operator+(Spec a, Spec b) { return {a.r + b.r, a.g + b.g, a.b + b.b}; }
PT_DEV Spec operator-(Spec a, Spec b) { return {a.r - b.r, a.g - b.g, a.b - b.b}; }
PT_DEV Spec operator*(Spec a, Spec b) { return {a.r * b.r, a.g * b.g, a.b * b.b}; }
PT_DEV Spec operator/(Spec a, Spec b) { return {a.r / b.r, a.g / b.g, a.b / b.b}; }
PT_DEV Spec operator*(Spec a, float s) { return {a.r * s, a.g * s, a.b * s}; }
PT_DEV Spec operator*(float s, Spec a) { return {a.r * s, a.g * s, a.b * s}; }
PT_DEV Spec operator/(Spec a, float s) { return {a.r / s, a.g / s, a.b / s}; }
PT_DEV bool is_black(Spec s) { return s.r == 0.f && s.g == 0.f && s.b == 0.f; }
PT_DEV float lum_y(Spec s) { return s.r * 0.212671f + s.g * 0.715160f + s.b * 0.072169f; }
PT_DEV float max_component(Spec s) { return fmaxf(fmaxf(s.r, s.g), s.b); }
PT_DEV Spec ssqrt(Spec s) { return {sqrtf(s.r), sqrtf(s.g), sqrtf(s.b)}; }
PT_DEV Spec lerps(Spec x, Spec y, float a) { return x * (1.0f - a) + y * a; }

}  // namespace ptrs
