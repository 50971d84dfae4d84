// BxDF lobes, Fresnel terms, the GGX distribution and the BSDF container on the device.
//   src/pathtracer/bxdf/mod.rs, bxdf/fresnel.rs, bxdf/microfacet.rs, material/disney.rs:57-170,
//   src/pathtracer/sampling.rs:96-126, src/pathtracer/bsdf.rs
#pragma once
#include "dev_math.cuh"

namespace ptrs {

PT_DEV float cos_theta(V3 w) { return w.z; }
PT_DEV float cos_2_theta(V3 w) { return w.z * w.z; }
PT_DEV float abs_cos_theta(V3 w) { return fabsf(w.z); }
PT_DEV float sin_2_theta(V3 w) { return fmaxf(0.0f, 1.0f - cos_2_theta(w)); }
PT_DEV float sin_theta(V3 w) { return sqrtf(sin_2_theta(w)); }
PT_DEV float tan_2_theta(V3 w) { return sin_2_theta(w) / cos_2_theta(w); }
PT_DEV float tan_theta(V3 w) { return sin_theta(w) / cos_theta(w); }
PT_DEV float cos_phi(V3 w) {
  float st = sin_theta(w);
  return st == 0.0f ? 1.0f : rclamp(w.x / st, -1.0f, 1.0f);
}
PT_DEV float sin_phi(V3 w) {  // returns 1.0 at the pole like the reference (bxdf/mod.rs:49-56)
  float st = sin_theta(w);
  return st == 0.0f ? 1.0f : rclamp(w.y / st, -1.0f, 1.0f);
}
PT_DEV float cos_2_phi(V3 w) { return cos_phi(w) * cos_phi(w); }
PT_DEV float sin_2_phi(V3 w) { return sin_phi(w) * sin_phi(w); }
PT_DEV bool same_hemisphere(V3 w, V3 wp) { return w.z * wp.z > 0.0f; }
PT_DEV V3 reflect(V3 wo, V3 n) { return -wo + 2.f * dot(wo, n) * n; }
PT_DEV bool refract(V3 wi, V3 n, float eta, V3* wt) {  // bxdf/mod.rs:73-89
  float cos_theta_i = dot(n, wi);
  float sin_2_theta_i = fmaxf(0.0f, 1.0f - cos_theta_i * cos_theta_i);
  float sin_2_theta_t = eta * eta * sin_2_theta_i;
  if (sin_2_theta_t > 1.0f) return false;
  float cos_theta_t = sqrtf(1.0f - sin_2_theta_t);
  *wt = eta * -wi + (eta * cos_theta_i - cos_theta_t) * n;
  return true;
}

enum : uint32_t {
  BSDF_REFLECTION = 1, BSDF_TRANSMISSION = 2, BSDF_DIFFUSE = 4, BSDF_GLOSSY = 8, BSDF_SPECULAR = 16, BSDF_ALL = 31
};

PT_DEV V2 concentric_sample_disk(V2 u) {  // sampling.rs:96-116
  float ox = 2.0f * u.x - 1.0f, oy = 2.0f * u.y - 1.0f;
  if (ox == 0.0f && oy == 0.0f) return V2{0.0f, 0.0f};
  float theta, r;
  if (fabsf(ox) > fabsf(oy)) {
    r = ox;
    theta = PT_FRAC_PI_4 * (oy / ox);
  } else {
    r = oy;
    theta = PT_FRAC_PI_2 - PT_FRAC_PI_4 * (ox / oy);
  }
  return V2{r * cos_small_angle(theta), r * sin_small_angle(theta)};
}
PT_DEV V3 cosine_sample_hemisphere(V2 u) {  // sampling.rs:118-122
  V2 d = concentric_sample_disk(u);
  float z = sqrtf(fmaxf(0.0f, 1.0f - d.x * d.x - d.y * d.y));
  return mk3(d.x, d.y, z);
}

PT_DEV float fr_dielectric(float cos_theta_i, float eta_i, float eta_t) {  // fresnel.rs:21-40
  cos_theta_i = rclamp(cos_theta_i, -1.0f, 1.0f);
  if (!(cos_theta_i > 0.0f)) {
    float tmp = eta_i;
    eta_i = eta_t;
    eta_t = tmp;
    cos_theta_i = fabsf(cos_theta_i);
  }
  float sin_theta_i = sqrtf(fmaxf(0.0f, 1.0f - cos_theta_i * cos_theta_i));
  float sin_theta_t = eta_i / eta_t * sin_theta_i;
  if (sin_theta_t >= 1.0f) return 1.0f;
  float cos_theta_t = sqrtf(fmaxf(0.0f, 1.0f - sin_theta_t * sin_theta_t));
  float r_parl = ((eta_t * cos_theta_i) - (eta_i * cos_theta_t)) / ((eta_t * cos_theta_i) + (eta_i * cos_theta_t));
  float r_perp = ((eta_i * cos_theta_i) - (eta_t * cos_theta_t)) / ((eta_i * cos_theta_i) + (eta_t * cos_theta_t));
  return (r_parl * r_parl + r_perp * r_perp) / 2.0f;
}
PT_DEV Spec fr_conductor(float cos_theta_i, Spec eta_i, Spec eta_t, Spec k) {  // fresnel.rs:42-64
  cos_theta_i = rclamp(cos_theta_i, -1.f, 1.f);
  Spec eta = eta_t / eta_i, etak = k / eta_i;
  float c2 = cos_theta_i * cos_theta_i;
  float s2 = 1.f - c2;
  Spec eta2 = eta * eta, etak2 = etak * etak;
  Spec t0 = eta2 - etak2 - sp(s2);
  Spec a2_plus_b2 = ssqrt(t0 * t0 + 4.f * eta2 * etak2);
  Spec t1 = a2_plus_b2 + sp(c2);
  Spec a = ssqrt(0.5f * (a2_plus_b2 + t0));
  Spec t2 = 2.f * cos_theta_i * a;
  Spec rs = (t1 - t2) / (t1 + t2);
  Spec t3 = c2 * a2_plus_b2 + sp(s2 * s2);
  Spec t4 = t2 * s2;
  Spec rp = rs * (t3 - t4) / (t3 + t4);
  return 0.5f * (rp + rs);
}
PT_DEV float schlick_weight(float c) {  // disney.rs:57-60
  float m = rclamp(1.0f - c, 0.0f, 1.0f);
  return (m * m) * (m * m) * m;
}

enum FresnelKind : int { FR_DIELECTRIC, FR_CONDUCTOR, FR_DISNEY, FR_NOOP };
enum LobeKind : int {
  LOBE_LAMBERT, LOBE_SPEC_REFL, LOBE_SPEC_TRANS, LOBE_FRESNEL_SPEC, LOBE_MF_REFL, LOBE_MF_TRANS, LOBE_FRESNEL_BLEND, LOBE_DISNEY_DIFFUSE
};

// One BxDF.  Field use by kind:
//   r: Lambert r / SpecRefl r / FresnelSpec r / MfRefl r / FresnelBlend rd / DisneyDiffuse r
//   t: SpecTrans t / FresnelSpec t / MfTrans t / FresnelBlend rs
//   fa, fb, fc: Fresnel params — conductor (eta_t, k), Disney (r0, {metallic, eta, -})
struct Lobe {
  int kind;
  int fresnel;
  Spec r, t;
  Spec fa, fb;
  float eta_a, eta_b;
  float alpha_x, alpha_y;
  int disney_g;  // separable G (DisneyMicrofacetDistribution, disney.rs:160-162)
};

// A shade<MAT> translation unit (k_shade.cu, -DPT_SHADE_MAT=<type>) only ever sees the lobes that material
// type creates (dev_shading.cuh compute_scattering_functions), so the lobe switches fold at compile time and
// the lobe functions can be inlined: the BSDF then lives in registers instead of local memory.
#ifdef PT_SHADE_MAT
#define PT_LOBE_FN __device__ __forceinline__
#if PT_SHADE_MAT == 0
#define PT_LOBE_MASK (1u << LOBE_LAMBERT)
#elif PT_SHADE_MAT == 1
#define PT_LOBE_MASK (1u << LOBE_SPEC_REFL)
#elif PT_SHADE_MAT == 2
#define PT_LOBE_MASK (1u << LOBE_FRESNEL_SPEC)
#elif PT_SHADE_MAT == 3
#define PT_LOBE_MASK (1u << LOBE_MF_REFL)
#elif PT_SHADE_MAT == 4
#define PT_LOBE_MASK (1u << LOBE_FRESNEL_BLEND)
#else
#define PT_LOBE_MASK ((1u << LOBE_DISNEY_DIFFUSE) | (1u << LOBE_MF_REFL))
#endif
#else
#define PT_LOBE_FN static __device__ __noinline__
#define PT_LOBE_MASK 0xffu
#endif
__host__ __device__ constexpr int pt_ctz(uint32_t m) { return (m & 1u) ? 0 : 1 + pt_ctz(m >> 1); }
__host__ __device__ constexpr int pt_popc(uint32_t m) { return m ? (int)(m & 1u) + pt_popc(m >> 1) : 0; }
__host__ __device__ constexpr int pt_top(uint32_t m) { return m > 1u ? 1 + pt_top(m >> 1) : 0; }
PT_DEV int lobe_kind(const Lobe& l) {
  constexpr uint32_t m = PT_LOBE_MASK;
  if (pt_popc(m) == 1) return pt_ctz(m);
  if (pt_popc(m) == 2) return l.kind == pt_ctz(m) ? pt_ctz(m) : pt_top(m);
  return l.kind;
}

PT_DEV uint32_t lobe_type(const Lobe& l) {
  switch (lobe_kind(l)) {
    case LOBE_LAMBERT: case LOBE_DISNEY_DIFFUSE: return BSDF_REFLECTION | BSDF_DIFFUSE;
    case LOBE_SPEC_REFL: return BSDF_REFLECTION | BSDF_SPECULAR;
    case LOBE_SPEC_TRANS: return BSDF_TRANSMISSION | BSDF_SPECULAR;
    case LOBE_FRESNEL_SPEC: return BSDF_REFLECTION | BSDF_TRANSMISSION | BSDF_SPECULAR;
    case LOBE_MF_REFL: case LOBE_FRESNEL_BLEND: return BSDF_REFLECTION | BSDF_GLOSSY;
    default: return BSDF_TRANSMISSION | BSDF_GLOSSY;
  }
}
PT_DEV bool lobe_matches(const Lobe& l, uint32_t flags) {
  uint32_t t = lobe_type(l);
  return (t & flags) == t;
}

PT_DEV Spec fresnel_eval(const Lobe& l, float cos_i) {
  switch (l.fresnel) {
    case FR_DIELECTRIC: return sp(fr_dielectric(cos_i, l.eta_a, l.eta_b));
    case FR_CONDUCTOR: return fr_conductor(fabsf(cos_i), sp(1.f), l.fa, l.fb);
    case FR_DISNEY: {  // disney.rs:128-136: lerp(dielectric(cos, 1, eta), schlick(r0), metallic)
      Spec schlick = lerps(l.fa, sp(1.f), schlick_weight(cos_i));
      return lerps(sp(fr_dielectric(cos_i, 1.f, l.fb.g)), schlick, l.fb.r);
    }
    default: return sp(1.0f);
  }
}

// TrowbridgeReitzDistribution, microfacet.rs:106-174
PT_DEV float ggx_d(const Lobe& l, V3 wh) {
  float t2 = tan_2_theta(wh);
  if (isinf(t2)) return 0.0f;
  float cos_4_theta = cos_2_theta(wh) * cos_2_theta(wh);
  float e = (cos_2_phi(wh) / (l.alpha_x * l.alpha_x) + sin_2_phi(wh) / (l.alpha_y * l.alpha_y)) * t2;
  return 1.0f / (PT_PI * l.alpha_x * l.alpha_y * cos_4_theta * (1.0f + e) * (1.0f + e));
}
PT_DEV float ggx_lambda(const Lobe& l, V3 w) {
  float abs_tan_theta = fabsf(tan_theta(w));
  if (isinf(abs_tan_theta)) return 0.0f;
  float alpha = sqrtf((cos_2_phi(w) * l.alpha_x * l.alpha_x) + (sin_2_phi(w) * l.alpha_y * l.alpha_y));
  float a2t2 = (alpha * abs_tan_theta) * (alpha * abs_tan_theta);
  return (-1.0f + sqrtf(1.0f + a2t2)) / 2.0f;
}
PT_DEV float ggx_g1(const Lobe& l, V3 w) { return 1.0f / (1.0f + ggx_lambda(l, w)); }
PT_DEV float ggx_g(const Lobe& l, V3 wo, V3 wi) {
  if (l.disney_g) return ggx_g1(l, wo) * ggx_g1(l, wi);
  return 1.0f / (1.0f + ggx_lambda(l, wo) + ggx_lambda(l, wi));
}
PT_DEV void trowbridge_reitz_sample_11(float cos_t, float u1, float u2, float* slope_x, float* slope_y) {  // microfacet.rs:32-81
  if (cos_t > 0.9999f) {
    float r = sqrtf(u1 / (1.f - u1));
    float phi = 6.28318530718f * u2;
    *slope_x = r * cos_small_angle(phi);
    *slope_y = r * sin_small_angle(phi);
    return;
  }
  float sin_t = sqrtf(fmaxf(0.0f, 1.f - cos_t * cos_t));
  float tan_t = sin_t / cos_t;
  float alpha = 1.f / tan_t;
  float g1 = 2.f / (1.f + sqrtf(1.f + 1.f / (alpha * alpha)));
  float a = 2.f * u1 / g1 - 1.f;
  float tmp = 1.f / (a * a - 1.f);
  if (tmp > 1e10f) tmp = 1e10f;
  float b = tan_t;
  float d = sqrtf(fmaxf(0.0f, b * b * tmp * tmp - (a * a - b * b) * tmp));
  float slope_x_1 = b * tmp - d, slope_x_2 = b * tmp + d;
  *slope_x = (a < 0.f || slope_x_2 > (1.f / tan_t)) ? slope_x_1 : slope_x_2;
  float s;
  if (u2 > 0.5f) {
    s = 1.f;
    u2 = 2.f * (u2 - 0.5f);
  } else {
    s = -1.f;
    u2 = 2.f * (0.5f - u2);
  }
  float z = (u2 * (u2 * (u2 * 0.27385f - 0.73369f) + 0.46341f)) / (u2 * (u2 * (u2 * 0.093073f + 0.309420f) - 1.000000f) + 0.597999f);
  *slope_y = s * z * sqrtf(1.f + *slope_x * *slope_x);
}
PT_DEV V3 ggx_sample_wh(const Lobe& l, V3 wo, V2 u) {  // microfacet.rs:83-104, 161-169
  bool flip = wo.z < 0.f;
  V3 w = flip ? -wo : wo;
  V3 ws = normalize(mk3(l.alpha_x * w.x, l.alpha_y * w.y, w.z));
  float slope_x = 0.f, slope_y = 0.f;
  trowbridge_reitz_sample_11(cos_theta(ws), u.x, u.y, &slope_x, &slope_y);
  float tmp = cos_phi(ws) * slope_x - sin_phi(ws) * slope_y;
  slope_y = sin_phi(ws) * slope_x + cos_phi(ws) * slope_y;
  slope_x = tmp;
  slope_x = l.alpha_x * slope_x;
  slope_y = l.alpha_y * slope_y;
  V3 wh = normalize(mk3(-slope_x, -slope_y, 1.f));
  return flip ? -wh : wh;
}
PT_DEV float ggx_pdf(const Lobe& l, V3 wo, V3 wh) { return ggx_d(l, wh) * ggx_g1(l, wo) * fabsf(dot(wo, wh)) / abs_cos_theta(wo); }
PT_DEV float roughness_to_alpha(float roughness) {  // microfacet.rs:119-128
  roughness = fmaxf(roughness, 1e-3f);
  float x = logf(roughness);
  return 1.62142f + 0.819955f * x + 0.1734f * x * x + 0.0171201f * x * x * x + 0.000640711f * x * x * x * x;
}
PT_DEV float pow5(float v) { return (v * v) * (v * v) * v; }

PT_LOBE_FN Spec lobe_f(const Lobe& l, V3 wo, V3 wi) {
  switch (lobe_kind(l)) {
    case LOBE_LAMBERT: return l.r * PT_FRAC_1_PI;
    case LOBE_DISNEY_DIFFUSE: {
      float fo = schlick_weight(abs_cos_theta(wo)), fi = schlick_weight(abs_cos_theta(wi));
      return l.r * PT_FRAC_1_PI * (1.f - fo / 2.f) * (1.f - fi / 2.f);
    }
    case LOBE_MF_REFL: {
      float cos_o = abs_cos_theta(wo), cos_i = abs_cos_theta(wi);
      V3 wh = wi + wo;
      if (cos_i == 0.f || cos_o == 0.f) return sp(0.f);
      if (wh.x == 0.f && wh.y == 0.f && wh.z == 0.f) return sp(0.f);
      wh = normalize(wh);
      Spec fr = fresnel_eval(l, dot(wi, wh));
      return l.r * ggx_d(l, wh) * ggx_g(l, wo, wi) * fr / (4.0f * cos_i * cos_o);
    }
    case LOBE_MF_TRANS: {
      if (same_hemisphere(wo, wi)) return sp(0.f);
      float cos_o = abs_cos_theta(wo), cos_i = abs_cos_theta(wi);
      if (cos_i == 0.f || cos_o == 0.f) return sp(0.f);
      float eta = cos_theta(wo) > 0.0f ? l.eta_b / l.eta_a : l.eta_a / l.eta_b;
      V3 wh = normalize(wo + wi * eta);
      if (wh.z < 0.0f) wh = -wh;
      if (dot(wo, wh) * dot(wi, wh) > 0.f) return sp(0.f);
      Spec fr = sp(fr_dielectric(dot(wo, wh), l.eta_a, l.eta_b));
      float sqrt_denom = dot(wo, wh) + eta * dot(wi, wh);
      float factor = 1.0f / eta;
      return (sp(1.f) - fr) * l.t *
             (ggx_d(l, wh) * ggx_g(l, wo, wi) * eta * eta * fabsf(dot(wi, wh)) * fabsf(dot(wo, wh)) * factor * factor /
              (cos_i * cos_o * sqrt_denom * sqrt_denom));
    }
    case LOBE_FRESNEL_BLEND: {
      Spec diffuse = (28.f / (23.f * PT_PI)) * l.r * (sp(1.f) - l.t) * (1.f - pow5(1.f - 0.5f * abs_cos_theta(wi))) *
                     (1.f - pow5(1.f - 0.5f * abs_cos_theta(wo)));
      V3 wh = wi + wo;
      if (is_zero3(wh)) return sp(0.f);
      wh = normalize(wh);
      Spec schlick = l.t + pow5(1.0f - dot(wi, wh)) * (sp(1.f) - l.t);
      Spec specular = ggx_d(l, wh) / (4.f * fabsf(dot(wi, wh)) * fmaxf(abs_cos_theta(wi), abs_cos_theta(wo))) * schlick;
      return diffuse + specular;
    }
    default: return sp(0.0f);
  }
}

PT_LOBE_FN float lobe_pdf(const Lobe& l, V3 wo, V3 wi) {
  switch (lobe_kind(l)) {
    case LOBE_LAMBERT: case LOBE_DISNEY_DIFFUSE: return same_hemisphere(wo, wi) ? abs_cos_theta(wi) * PT_FRAC_1_PI : 0.0f;
    case LOBE_MF_REFL: {
      if (!same_hemisphere(wo, wi)) return 0.f;
      V3 wh = normalize(wo + wi);
      return ggx_pdf(l, wo, wh) / (4.f * dot(wo, wh));
    }
    case LOBE_MF_TRANS: {  // microfacet.rs:363-383 (rejects the opposite hemisphere, as the reference does)
      if (!same_hemisphere(wo, wi)) return 0.f;
      float eta = cos_theta(wo) > 0.f ? l.eta_a / l.eta_b : l.eta_b / l.eta_a;
      V3 wh = normalize(wo + wi * eta);
      if (dot(wo, wh) * dot(wi, wh) > 0.f) return 0.f;
      float sqrt_denom = dot(wo, wh) + eta * dot(wi, wh);
      float dwh_dwi = fabsf((eta * eta * dot(wi, wh)) / (sqrt_denom * sqrt_denom));
      return ggx_pdf(l, wo, wh) * dwh_dwi;
    }
    case LOBE_FRESNEL_BLEND: {
      if (!same_hemisphere(wo, wi)) return 0.f;
      V3 wh = normalize(wo + wi);
      float pdf_wh = ggx_pdf(l, wo, wh);
      return 0.5f * (abs_cos_theta(wi) * PT_FRAC_1_PI + pdf_wh / (4.f * dot(wo, wh)));
    }
    default: return 0.0f;
  }
}

// BxDFInterface::sample_f; *sampled_type only changes for FresnelSpecular (fresnel.rs:254-288)
PT_LOBE_FN Spec lobe_sample_f(const Lobe& l, V3 wo, V3* wi, V2 u, float* pdf, uint32_t* sampled_type) {
  switch (lobe_kind(l)) {
    case LOBE_LAMBERT: case LOBE_DISNEY_DIFFUSE: {
      *wi = cosine_sample_hemisphere(u);
      if (wo.z < 0.0f) wi->z *= -1.0f;
      *pdf = lobe_pdf(l, wo, *wi);
      return lobe_f(l, wo, *wi);
    }
    case LOBE_SPEC_REFL: {
      *wi = mk3(-wo.x, -wo.y, wo.z);
      *pdf = 1.0f;
      return fresnel_eval(l, cos_theta(*wi)) * l.r / abs_cos_theta(*wi);
    }
    case LOBE_SPEC_TRANS: {
      bool entering = cos_theta(wo) > 0.0f;
      float eta_i = entering ? l.eta_a : l.eta_b, eta_t = entering ? l.eta_b : l.eta_a;
      if (!refract(wo, face_forward(mk3(0.f, 0.f, 1.f), wo), eta_i / eta_t, wi)) return sp(0.0f);
      *pdf = 1.0f;
      Spec ft = l.t * (sp(1.0f) - sp(fr_dielectric(cos_theta(*wi), l.eta_a, l.eta_b)));
      ft = ft * ((eta_i * eta_i) / (eta_t * eta_t));
      return ft / abs_cos_theta(*wi);
    }
    case LOBE_FRESNEL_SPEC: {
      float fr = fr_dielectric(cos_theta(wo), l.eta_a, l.eta_b);
      if (u.x < fr) {
        *wi = mk3(-wo.x, -wo.y, wo.z);
        *sampled_type = BSDF_REFLECTION | BSDF_SPECULAR;
        *pdf = fr;
        return fr * l.r / abs_cos_theta(*wi);
      } else {
        bool entering = cos_theta(wo) > 0.0f;
        float eta_i = entering ? l.eta_a : l.eta_b, eta_t = entering ? l.eta_b : l.eta_a;
        if (!refract(wo, face_forward(mk3(0.f, 0.f, 1.f), wo), eta_i / eta_t, wi)) return sp(0.0f);
        Spec ft = l.t * (sp(1.0f) - sp(fr));
        ft = ft * ((eta_i * eta_i) / (eta_t * eta_t));
        *sampled_type = BSDF_TRANSMISSION | BSDF_SPECULAR;
        *pdf = 1.0f - fr;
        return ft / abs_cos_theta(*wi);
      }
    }
    case LOBE_MF_REFL: {
      if (wo.z == 0.f) return sp(0.f);
      V3 wh = ggx_sample_wh(l, wo, u);
      if (dot(wo, wh) < 0.f) return sp(0.f);
      *wi = reflect(wo, wh);
      if (!same_hemisphere(wo, *wi)) return sp(0.f);
      *pdf = ggx_pdf(l, wo, wh) / (4.f * dot(wo, wh));
      return lobe_f(l, wo, *wi);
    }
    case LOBE_MF_TRANS: {
      if (wo.z == 0.f) return sp(0.f);
      V3 wh = ggx_sample_wh(l, wo, u);
      if (dot(wo, wh) < 0.f) return sp(0.f);
      float eta = cos_theta(wo) > 0.f ? l.eta_a / l.eta_b : l.eta_b / l.eta_a;
      if (!refract(wo, wh, eta, wi)) return sp(0.f);
      *pdf = lobe_pdf(l, wo, *wi);
      return lobe_f(l, wo, *wi);
    }
    default: {  // LOBE_FRESNEL_BLEND, microfacet.rs:433-458
      V2 uu = u;
      if (uu.x < 0.5f) {
        uu.x = fminf(2.f * uu.x, PT_ONE_MINUS_EPSILON);
        *wi = cosine_sample_hemisphere(uu);
        if (wo.z < 0.f) wi->z *= -1.f;
      } else {
        uu.x = fminf(2.f * (uu.x - 0.5f), PT_ONE_MINUS_EPSILON);
        V3 wh = ggx_sample_wh(l, wo, uu);
        *wi = reflect(wo, wh);
        if (!same_hemisphere(wo, *wi)) return sp(0.f);
      }
      *pdf = lobe_pdf(l, wo, *wi);
      return lobe_f(l, wo, *wi);
    }
  }
}

// BSDF (bsdf.rs:8-222).  No material of the reference adds more than two lobes (Disney).
#define PT_MAX_LOBES 2
struct Bsdf {
  float eta;
  V3 ns, ng, ss, ts;
  int n;
  Lobe lobes[PT_MAX_LOBES];
};
PT_DEV V3 world_to_local(const Bsdf& b, V3 v) { return mk3(dot(v, b.ss), dot(v, b.ts), dot(v, b.ns)); }
PT_DEV V3 local_to_world(const Bsdf& b, V3 v) {
  return mk3(b.ss.x * v.x + b.ts.x * v.y + b.ns.x * v.z, b.ss.y * v.x + b.ts.y * v.y + b.ns.y * v.z, b.ss.z * v.x + b.ts.z * v.y + b.ns.z * v.z);
}
PT_DEV int bsdf_num_components(const Bsdf& b, uint32_t flags) {
  int c = 0;
  for (int i = 0; i < PT_MAX_LOBES; ++i)
    if (i < b.n && lobe_matches(b.lobes[i], flags)) ++c;
  return c;
}

PT_DEV Spec bsdf_f(const Bsdf& b, V3 wo_w, V3 wi_w, uint32_t flags) {  // bsdf.rs:150-187
  V3 wi = world_to_local(b, wi_w), wo = world_to_local(b, wo_w);
  if (wo.z == 0.0f) return sp(0.0f);
  bool refl = dot(wi_w, b.ng) * dot(wo_w, b.ng) > 0.0f;
  Spec f = sp(0.0f);
  for (int i = 0; i < PT_MAX_LOBES; ++i)
    if (i < b.n && lobe_matches(b.lobes[i], flags)) {
      uint32_t t = lobe_type(b.lobes[i]);
      if ((refl && (t & BSDF_REFLECTION)) || (!refl && (t & BSDF_TRANSMISSION))) f = f + lobe_f(b.lobes[i], wo, wi);
    }
  return f;
}
PT_DEV float bsdf_pdf(const Bsdf& b, V3 wo_w, V3 wi_w, uint32_t flags) {  // bsdf.rs:189-222
  if (b.n == 0) return 0.0f;
  V3 wo = world_to_local(b, wo_w), wi = world_to_local(b, wi_w);
  if (wo.z == 0.0f) return 0.0f;
  float pdf = 0.0f;
  int matching = 0;
  for (int i = 0; i < PT_MAX_LOBES; ++i)
    if (i < b.n && lobe_matches(b.lobes[i], flags)) {
      matching += 1;
      pdf += lobe_pdf(b.lobes[i], wo, wi);
    }
  return matching > 0 ? pdf / (float)matching : 0.0f;
}
PT_DEV Spec bsdf_sample_f(const Bsdf& b, V3 wo_w, V3* wi_w, V2 u, float* pdf, uint32_t type, uint32_t* sampled_type) {  // bsdf.rs:66-148
  int matching = bsdf_num_components(b, type);
  if (matching == 0) {
    *pdf = 0.0f;
    *sampled_type = 0;
    return sp(0.0f);
  }
  unsigned long long c64 = (unsigned long long)floorf(u.x * (float)matching);
  int comp = (int)(c64 < (unsigned long long)(matching - 1) ? c64 : (unsigned long long)(matching - 1));
  int sel = 0, count = comp;
  for (int i = 0; i < PT_MAX_LOBES; ++i)
    if (i < b.n && lobe_matches(b.lobes[i], type)) {
      if (count == 0) {
        sel = i;
        break;
      }
      count -= 1;
    }
  // A material with one lobe kind has at most one lobe, so sel == 0: b.lobes indexed with the run-time `sel` would keep
  // the whole BSDF in local memory.  Disney's two lobes keep the indexed access.
  const Lobe& lobe = pt_popc(PT_LOBE_MASK) == 1 ? b.lobes[0] : b.lobes[sel];
  V2 u_remapped{(u.x * (float)matching) - (float)comp, u.y};
  V3 wi = mk3(0, 0, 0);
  V3 wo = world_to_local(b, wo_w);
  *pdf = 0.0f;
  *sampled_type = lobe_type(lobe);
  Spec f = lobe_sample_f(lobe, wo, &wi, u_remapped, pdf, sampled_type);
  if (*pdf == 0.0f) {
    *sampled_type = 0;
    return sp(0.0f);
  }
  *wi_w = local_to_world(b, wi);
  const bool spec = (lobe_type(lobe) & BSDF_SPECULAR) != 0;
  if (!spec && matching > 1)
    for (int i = 0; i < PT_MAX_LOBES; ++i)
      if (i < b.n && i != sel && lobe_matches(b.lobes[i], type)) *pdf += lobe_pdf(b.lobes[i], wo, wi);
  if (matching > 1) *pdf /= (float)matching;
  if (!spec && matching > 1) {
    bool refl = dot(*wi_w, b.ng) * dot(wo_w, b.ng) > 0.0f;
    f = sp(0.0f);
    for (int i = 0; i < PT_MAX_LOBES; ++i)
      if (i < b.n && lobe_matches(b.lobes[i], type)) {
        uint32_t t = lobe_type(b.lobes[i]);
        if ((refl && (t & BSDF_REFLECTION)) || (!refl && (t & BSDF_TRANSMISSION))) f = f + lobe_f(b.lobes[i], wo, wi);
      }
  }
  return f;
}

}  // namespace ptrs
