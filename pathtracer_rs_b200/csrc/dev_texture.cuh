// Texture evaluation on the device: src/pathtracer/texture.rs (ConstantTexture :15-29, UVMap :31-54,
// CheckerTexture :56-89, ImageTexture :185-192, MIPMap::{texel, triangle, lookup, lookup_width}).
#pragma once
#include "dev_scene.cuh"

namespace ptrs {

// what Texture::evaluate reads from the SurfaceMediumInteraction
struct TexCoord {
  float u, v;
  float dudx, dvdx, dudy, dvdy;
};

// The lookup chain returns its texel by value and indexes no array, so nothing in it needs an address. A shade
// translation unit (-DPT_SHADE_MAT) inlines it and keeps the texel in registers, with no local-memory frame; elsewhere
// (the alpha test of the traversal kernels, the miss and resolve kernels) tex_eval_slow and mip_lookup_width stay calls.
// A texture has 1 or 3 channels; a 1-channel texel is (v, 0, 0).
#ifdef PT_SHADE_MAT
#define PT_TEX_FN __device__ __forceinline__
#else
#define PT_TEX_FN static __device__ __noinline__
#endif

PT_DEV Spec mip_texel(const DevScene& sc, const PtrsMipMap& mm, int level, int s, int t) {  // texture.rs:245-273
  const int W = mm.width[level], H = mm.height[level], C = mm.channels;
  if (mm.wrap == PTRS_WRAP_REPEAT) {
    // abs_mod(a, b) == a & (b - 1) for power-of-two b (MIP levels are powers of two after MIPMap::new's
    // resample, texture.rs:285-295): avoids two integer divisions per texel
    s = (W & (W - 1)) == 0 ? (s & (W - 1)) : abs_mod(s, W);
    t = (H & (H - 1)) == 0 ? (t & (H - 1)) : abs_mod(t, H);
  } else if (mm.wrap == PTRS_WRAP_BLACK) {
    if (s < 0 || s >= W || t < 0 || t >= H) return sp(0.f);
  } else {
    s = min(max(s, 0), W - 1);
    t = min(max(t, 0), H - 1);
  }
  const float* p = sc.texels + mm.level_offset[level] + ((size_t)t * W + s) * C;
  if (C == 3) return sp(__ldg(p), __ldg(p + 1), __ldg(p + 2));
  return sp(__ldg(p), 0.f, 0.f);
}

PT_DEV float mip_bilerp(float a, float b, float c, float e, float ds, float dt) {
  return ((a * (1.0f - ds) * (1.0f - dt) + b * (1.0f - ds) * dt) + c * ds * (1.0f - dt)) + e * ds * dt;
}
PT_DEV Spec mip_triangle(const DevScene& sc, const PtrsMipMap& mm, int level, float su, float tv) {  // texture.rs:413-429
  level = min(max(level, 0), mm.n_levels - 1);
  float s = su * (float)mm.width[level] - 0.5f;
  float t = tv * (float)mm.height[level] - 0.5f;
  float s0f = floorf(s), t0f = floorf(t);
  float ds = s - s0f, dt = t - t0f;
  int s0 = (int)s0f, t0 = (int)t0f;
  const Spec a = mip_texel(sc, mm, level, s0, t0);
  const Spec b = mip_texel(sc, mm, level, s0, t0 + 1);
  const Spec c = mip_texel(sc, mm, level, s0 + 1, t0);
  const Spec e = mip_texel(sc, mm, level, s0 + 1, t0 + 1);
  const bool rgb = mm.channels == 3;
  return sp(mip_bilerp(a.r, b.r, c.r, e.r, ds, dt), rgb ? mip_bilerp(a.g, b.g, c.g, e.g, ds, dt) : 0.f,
            rgb ? mip_bilerp(a.b, b.b, c.b, e.b, ds, dt) : 0.f);
}

// One level, or the lerp of two adjacent levels: mip_triangle is written out twice, not three times.
PT_TEX_FN Spec mip_lookup_width(const DevScene& sc, const PtrsMipMap& mm, float s, float t, float width) {  // texture.rs:447-464
  const int n = mm.n_levels;
  float level = (float)n - 1.0f + log2f(fmaxf(width, 1e-8f));
  const bool one = level < 0.0f || level >= (float)(n - 1);
  const float il = floorf(level);
  const Spec a = mip_triangle(sc, mm, one ? (level < 0.0f ? 0 : n - 1) : (int)il, s, t);
  if (one) return a;
  const float delta = level - il;
  const Spec b = mip_triangle(sc, mm, (int)il + 1, s, t);
  const bool rgb = mm.channels == 3;
  return sp(a.r * (1.0f - delta) + b.r * delta, rgb ? a.g * (1.0f - delta) + b.g * delta : 0.f, rgb ? a.b * (1.0f - delta) + b.b * delta : 0.f);
}

PT_TEX_FN Spec tex_eval_slow(const DevScene& sc, int tex_id, const TexCoord& tc) {
  const PtrsTexture& t = sc.textures[tex_id];
  if (t.type == PTRS_TEX_CHECKER) {
    float s = t.su * tc.u + t.du, tt = t.sv * tc.v + t.dv;
    float s_idx = s - floorf(s), t_idx = tt - floorf(tt);
    bool second = (s_idx <= 0.5f && t_idx <= 0.5f) || (s_idx >= 0.5f && t_idx >= 0.5f);
    return second ? sp(t.v2[0], t.v2[1], t.v2[2]) : sp(t.v1[0], t.v1[1], t.v1[2]);
  }
  float dsdx = t.su * tc.dudx, dtdx = t.sv * tc.dvdx, dsdy = t.su * tc.dudy, dtdy = t.sv * tc.dvdy;
  float s = t.su * tc.u + t.du, tt = t.sv * tc.v + t.dv;
  float width = fmaxf(fmaxf(fabsf(dsdx), fabsf(dtdx)), fmaxf(fabsf(dsdy), fabsf(dtdy)));  // MIPMap::lookup
  return mip_lookup_width(sc, sc.mipmaps[t.mip], s, tt, width);
}
// ConstantTexture (the common case: every Mitsuba rgb / float parameter) is resolved inline
PT_DEV Spec tex_eval(const DevScene& sc, int tex_id, const TexCoord& tc) {
  const PtrsTexture* t = sc.textures + tex_id;
  if (__ldg(&t->type) == PTRS_TEX_CONSTANT) return sp(__ldg(&t->v1[0]), __ldg(&t->v1[1]), __ldg(&t->v1[2]));
  return tex_eval_slow(sc, tex_id, tc);
}
PT_DEV float tex_f32(const DevScene& sc, int id, const TexCoord& tc) { return tex_eval(sc, id, tc).r; }
PT_DEV Spec tex_spec(const DevScene& sc, int id, const TexCoord& tc) { return tex_eval(sc, id, tc); }

}  // namespace ptrs
