// Surface interaction reconstruction, materials and lights on the device.
//   Triangle::intersect geometry block   src/pathtracer/shape.rs:187-356
//   Triangle::{sample, pdf_at_point}      shape.rs:62-72, 541-578
//   Interaction / SurfaceMediumInteraction src/pathtracer/interaction.rs
//   Material::compute_scattering_functions src/pathtracer/material/{mod,metal,substrate,disney}.rs
//   Light::{sample_li, pdf_li, le}         src/pathtracer/light.rs, sampling.rs:128-230
#pragma once
#include "dev_accel.cuh"
#include "dev_bxdf.cuh"

namespace ptrs {

#define PT_SHADOW_EPSILON 0.0001f

struct Inter {  // Interaction, interaction.rs:9-15
  V3 p, p_error, n;
};
PT_DEV void spawn_ray(const Inter& it, V3 d, V3* o) { *o = offset_ray_origin(it.p, it.p_error, it.n, d); }  // interaction.rs:32-39
// interaction.rs:50-59: un-normalised segment, t_max = 1 - SHADOW_EPSILON
PT_DEV void spawn_ray_to_it(const Inter& a, const Inter& b, V3* o, V3* d) {
  V3 origin = offset_ray_origin(a.p, a.p_error, a.n, b.p - a.p);
  V3 target = offset_ray_origin(b.p, b.p_error, b.n, origin - b.p);
  *o = origin;
  *d = target - origin;
}

#ifdef PT_SHADE_MAT
#define PT_RECON_FN __device__ __forceinline__
#else
#define PT_RECON_FN static __device__ __noinline__
#endif

struct SurfInter {  // the fields of SurfaceMediumInteraction the path integrator reads
  Inter g;          // general {p, p_error, n}
  V3 wo;
  V2 uv;
  V3 dpdu, dpdv;             // geometric partials
  V3 sh_n, sh_dpdu, sh_dpdv;  // shading frame
  float dudx, dvdx, dudy, dvdy;
  int prim;
};

struct __align__(32) F8s {
  float4 a, b;
};
PT_DEV F8s ld256_nc(const F8s* p) {  // LDG.E.256 through the read-only path
  F8s v;
  asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(v.a.x), "=f"(v.a.y), "=f"(v.a.z), "=f"(v.a.w), "=f"(v.b.x), "=f"(v.b.y), "=f"(v.b.z), "=f"(v.b.w)
      : "l"(p));
  return v;
}
PT_DEV V3 load3(const float* base, uint32_t i) { return mk3(__ldg(base + 3 * (size_t)i), __ldg(base + 3 * (size_t)i + 1), __ldg(base + 3 * (size_t)i + 2)); }

// Rebuilds what Triangle::intersect stored for the accepted hit (prim, b0, b1, b2).
PT_RECON_FN void reconstruct_hit(const DevScene& sc, int prim, float b0, float b1, float b2, V3 ray_d, SurfInter* si) {
  const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim), v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1),
               v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
  const V3 p0 = mk3(v0), p1 = mk3(v1), p2 = mk3(v2);
  const uint32_t flags = __float_as_uint(v2.w) & 0xffu;
  V2 uv[3];
  // the triangle's shading attributes come from its own 64-byte record (dev_scene.cuh tri_shade): two 32-byte loads that
  // depend on the primitive id only, instead of the index triple and up to fifteen gathers behind it
  const F8s sb = ld256_nc(reinterpret_cast<const F8s*>(sc.tri_shade + 4 * (size_t)prim) + 1);
  uv[0] = V2{sb.a.y, sb.a.z};
  uv[1] = V2{sb.a.w, sb.b.x};
  uv[2] = V2{sb.b.y, sb.b.z};
  V3 dpdu, dpdv;
  tri_partials(p0, p1, p2, uv, &dpdu, &dpdv);
  float x_abs_sum = fabsf(b0 * p0.x) + fabsf(b1 * p1.x) + fabsf(b2 * p2.x);
  float y_abs_sum = fabsf(b0 * p0.y) + fabsf(b1 * p1.y) + fabsf(b2 * p2.y);
  float z_abs_sum = fabsf(b0 * p0.z) + fabsf(b1 * p1.z) + fabsf(b2 * p2.z);
  si->g.p_error = gamma_n(7) * mk3(x_abs_sum, y_abs_sum, z_abs_sum);
  si->g.p = b0 * p0 + b1 * p1 + b2 * p2;
  si->uv = V2{b0 * uv[0].x + b1 * uv[1].x + b2 * uv[2].x, b0 * uv[0].y + b1 * uv[1].y + b2 * uv[2].y};
  si->wo = -ray_d;
  si->dpdu = dpdu;
  si->dpdv = dpdv;
  si->prim = prim;
  si->dudx = si->dvdx = si->dudy = si->dvdy = 0.f;
  V3 dp02 = p0 - p2, dp12 = p1 - p2;
  si->g.n = normalize(cross(dp02, dp12));
  si->sh_n = si->g.n;
  si->sh_dpdu = dpdu;
  si->sh_dpdv = dpdv;
  const bool has_n = flags & PTRS_MESH_HAS_NORMAL, has_s = flags & PTRS_MESH_HAS_TANGENT;
  if (has_n || has_s) {
    V3 ns;
    if (has_n) {
      const F8s sa = ld256_nc(reinterpret_cast<const F8s*>(sc.tri_shade + 4 * (size_t)prim));  // same 64-byte line as sb
      ns = b0 * mk3(sa.a.x, sa.a.y, sa.a.z) + b1 * mk3(sa.a.w, sa.b.x, sa.b.y) + b2 * mk3(sa.b.z, sa.b.w, sb.a.x);
      if (norm_squared(ns) > 0.0f) ns = normalize(ns);
      else ns = si->g.n;
    } else {
      ns = si->g.n;
    }
    V3 ss;
    if (has_s) {
      const uint4 idx = __ldg(sc.tri_index + prim);  // tangents (glTF only) stay per vertex
      ss = b0 * load3(sc.tangent, idx.x) + b1 * load3(sc.tangent, idx.y) + b2 * load3(sc.tangent, idx.z);
      if (norm_squared(ss) > 0.0f) ss = normalize(ss);
      else ss = normalize(dpdu);
    } else {
      ss = normalize(dpdu);
    }
    V3 ts = cross(ss, ns);
    if (norm_squared(ts) > 0.0f) {
      ts = normalize(ts);
      ss = cross(ts, ns);
    } else {
      coordinate_system(ns, &ss, &ts);
    }
    // set_shading_geometry(ss, ts, .., orientation_is_authoritative = true), interaction.rs:194-214
    si->sh_n = normalize(cross(ss, ts));
    si->g.n = face_forward(si->g.n, si->sh_n);
    si->sh_dpdu = ss;
    si->sh_dpdv = ts;
  }
}

// camera-ray differentials carried to the first hit (interaction.rs:216-281)
struct RayDiff {
  V3 rx_o, ry_o, rx_d, ry_d;
};
PT_DEV void compute_differentials(SurfInter* si, const RayDiff& rd) {
  const V3 n = si->g.n, p = si->g.p;
  float d = dot(n, p);
  float tx = -(dot(n, rd.rx_o) - d) / dot(n, rd.rx_d);
  if (isinf(tx) || tx != tx) return;
  V3 px = rd.rx_o + tx * rd.rx_d;
  float ty = -(dot(n, rd.ry_o) - d) / dot(n, rd.ry_d);
  if (isinf(ty) || ty != ty) return;
  V3 py = rd.ry_o + ty * rd.ry_d;
  int d0, d1;
  if (fabsf(n.x) > fabsf(n.y) && fabsf(n.x) > fabsf(n.y)) {  // sic, interaction.rs:241
    d0 = 1;
    d1 = 2;
  } else if (fabsf(n.y) > fabsf(n.z)) {
    d0 = 0;
    d1 = 2;
  } else {
    d0 = 0;
    d1 = 1;
  }
  float a00 = comp(si->dpdu, d0), a01 = comp(si->dpdv, d0), a10 = comp(si->dpdu, d1), a11 = comp(si->dpdv, d1);
  float bx0 = comp(px, d0) - comp(p, d0), bx1 = comp(px, d1) - comp(p, d1);
  float by0 = comp(py, d0) - comp(p, d0), by1 = comp(py, d1) - comp(p, d1);
  if (!solve_linear_system_2x2(a00, a01, a10, a11, bx0, bx1, &si->dudx, &si->dvdx)) si->dudx = si->dvdx = 0.0f;
  if (!solve_linear_system_2x2(a00, a01, a10, a11, by0, by1, &si->dudy, &si->dvdy)) si->dudy = si->dvdy = 0.0f;
}

PT_DEV TexCoord tc_of(const SurfInter& si) { return TexCoord{si.uv.x, si.uv.y, si.dudx, si.dvdx, si.dudy, si.dvdy}; }

PT_DEV void normal_mapping(const DevScene& sc, int tex, SurfInter* si) {  // material/mod.rs:39-79
  const V3 c0 = si->sh_dpdu, c1 = si->sh_dpdv, c2 = si->sh_n;
  const Spec o = tex_eval(sc, tex, tc_of(*si));
  V3 tn = normalize(mk3(o.r, o.g, o.b));
  V3 ns = normalize(mk3(c0.x * tn.x + c1.x * tn.y + c2.x * tn.z, c0.y * tn.x + c1.y * tn.y + c2.y * tn.z, c0.z * tn.x + c1.z * tn.y + c2.z * tn.z));
  V3 ss = si->sh_dpdu;
  V3 ts = cross(ss, ns);
  if (norm_squared(ts) > 0.0f) {
    ts = normalize(ts);
    ss = cross(ts, ns);
  } else {
    coordinate_system(ns, &ss, &ts);
  }
  si->sh_n = ns;
  si->sh_dpdu = ss;
  si->sh_dpdv = ts;
}

PT_DEV void bsdf_init(Bsdf* b, const SurfInter& si, float eta) {  // BSDF::new, bsdf.rs:20-34
  b->eta = eta;
  b->ns = si.sh_n;
  b->ss = normalize(si.sh_dpdu);
  b->ng = si.g.n;
  b->ts = cross(b->ns, b->ss);
  b->n = 0;
}
PT_DEV float sqr(float x) { return x * x; }

// returns false when the material leaves si.bsdf = None (Glass with black r and t, mod.rs:229-231)
template <int MAT>
PT_DEV bool compute_scattering_functions(const DevScene& sc, const PtrsMaterial& m, SurfInter* si, Bsdf* bsdf) {
  if (m.normal_map >= 0) normal_mapping(sc, m.normal_map, si);
  const TexCoord tc = tc_of(*si);
  Lobe& l0 = bsdf->lobes[0];
  if (MAT == PTRS_MAT_MATTE) {
    bsdf_init(bsdf, *si, 1.0f);
    l0.kind = LOBE_LAMBERT;
    l0.r = tex_spec(sc, m.tex[0], tc);
    bsdf->n = 1;
    return true;
  } else if (MAT == PTRS_MAT_MIRROR) {
    bsdf_init(bsdf, *si, 1.0f);
    l0.kind = LOBE_SPEC_REFL;
    l0.fresnel = FR_NOOP;
    l0.r = sp(1.0f);
    bsdf->n = 1;
    return true;
  } else if (MAT == PTRS_MAT_GLASS) {
    float eta = tex_f32(sc, m.tex[2], tc);
    Spec r = tex_spec(sc, m.tex[0], tc), t = tex_spec(sc, m.tex[1], tc);
    bsdf_init(bsdf, *si, eta);
    if (is_black(r) && is_black(t)) return false;
    l0.kind = LOBE_FRESNEL_SPEC;
    l0.r = r;
    l0.t = t;
    l0.eta_a = 1.0f;
    l0.eta_b = eta;
    bsdf->n = 1;
    return true;
  } else if (MAT == PTRS_MAT_METAL) {
    bsdf_init(bsdf, *si, 1.0f);
    float u_rough = tex_f32(sc, m.tex[3], tc), v_rough = tex_f32(sc, m.tex[4], tc);
    if (m.remap_roughness) {
      u_rough = roughness_to_alpha(u_rough);
      v_rough = roughness_to_alpha(v_rough);
    }
    l0.kind = LOBE_MF_REFL;
    l0.r = tex_spec(sc, m.tex[2], tc);
    l0.alpha_x = fmaxf(u_rough, 0.001f);
    l0.alpha_y = fmaxf(v_rough, 0.001f);
    l0.disney_g = 0;
    l0.fresnel = FR_CONDUCTOR;
    l0.fa = tex_spec(sc, m.tex[0], tc);
    l0.fb = tex_spec(sc, m.tex[1], tc);
    bsdf->n = 1;
    return true;
  } else if (MAT == PTRS_MAT_SUBSTRATE) {
    bsdf_init(bsdf, *si, 1.0f);
    Spec d = tex_spec(sc, m.tex[0], tc), s = tex_spec(sc, m.tex[1], tc);
    float rough_u = tex_f32(sc, m.tex[2], tc), rough_v = tex_f32(sc, m.tex[3], tc);
    if (!is_black(d) || is_black(s)) {  // sic, substrate.rs:55
      if (m.remap_roughness) {
        rough_u = roughness_to_alpha(rough_u);
        rough_v = roughness_to_alpha(rough_v);
      }
      l0.kind = LOBE_FRESNEL_BLEND;
      l0.r = d;
      l0.t = s;
      l0.alpha_x = fmaxf(rough_u, 0.001f);
      l0.alpha_y = fmaxf(rough_v, 0.001f);
      l0.disney_g = 0;
      bsdf->n = 1;
    }
    return true;
  } else {  // PTRS_MAT_DISNEY, disney.rs:172-263
    bsdf_init(bsdf, *si, 1.0f);
    Spec c = tex_spec(sc, m.tex[0], tc);
    float metallic_weight = tex_f32(sc, m.tex[1], tc);
    float e = tex_f32(sc, m.tex[2], tc);
    float diffuse_weight = (1.0f - metallic_weight) * (1.0f - 0.0f);
    float rough = tex_f32(sc, m.tex[3], tc);
    float lum = lum_y(c);
    Spec c_tint = lum > 0.0f ? c / lum : sp(1.0f);
    int k = 0;
    if (diffuse_weight > 0.0f) {
      Lobe& ld = bsdf->lobes[k++];
      ld.kind = LOBE_DISNEY_DIFFUSE;
      ld.r = diffuse_weight * c;
    }
    float ax = fmaxf(0.001f, sqr(rough) / 1.0f), ay = fmaxf(0.001f, sqr(rough) * 1.0f);
    float r0 = sqr(e - 1.0f) / sqr(e + 1.0f);  // schlick_r0_from_eta, mod.rs:100-102
    Spec c_spec_0 = lerps(r0 * lerps(sp(1.f), c_tint, 0.0f), c, metallic_weight);
    Lobe& ls = bsdf->lobes[k++];
    ls.kind = LOBE_MF_REFL;
    ls.r = sp(1.f);
    ls.alpha_x = fmaxf(ax, 0.001f);
    ls.alpha_y = fmaxf(ay, 0.001f);
    ls.disney_g = 1;
    ls.fresnel = FR_DISNEY;
    ls.fa = c_spec_0;
    ls.fb = sp(metallic_weight, e, 0.f);
    bsdf->n = k;
    return true;
  }
}

// ---- lights ----------------------------------------------------------------------------------------
PT_DEV V3 xform_vec(const float* m, V3 v) {
  return mk3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z);
}
PT_DEV size_t find_interval_cdf(const float* __restrict__ cdf, size_t size, float u) {  // math.rs:186-201
  size_t first = 0, len = size;
  while (len > 0) {
    size_t half = len >> 1, middle = first + half;
    if (__ldg(cdf + middle) <= u) {
      first = middle + 1;
      len -= half + 1;
    } else {
      len = half;
    }
  }
  size_t r = first - 1, hi = size - 2;
  return r > hi ? hi : r;
}
// find_interval restricted to the guide bracket [lo, hi]: the predicate cdf[i] <= u is monotone in i, so the
// partition point found inside the bracket is the one the full search finds
PT_DEV void pt_prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
PT_DEV size_t find_interval_guided(const float* __restrict__ cdf, size_t size, float u, const uint32_t* __restrict__ guide, uint32_t K,
                                   const float* __restrict__ func_hint = nullptr) {
  uint32_t k = (uint32_t)(u * (float)K);
  if (k > K - 1u) k = K - 1u;
  size_t first = __ldg(guide + k), len = __ldg(guide + k + 1) - first;
  // the bracket is known: start fetching the lines the search, the interval ends and the density will read, so the
  // dependent loads below meet them in L1 instead of each paying an L2 round trip
  pt_prefetch_l1(cdf + (first > 0 ? first - 1 : 0));
  if (func_hint) pt_prefetch_l1(func_hint + (first > 0 ? first - 1 : 0));
  while (len > 0) {
    size_t half = len >> 1, middle = first + half;
    if (__ldg(cdf + middle) <= u) {
      first = middle + 1;
      len -= half + 1;
    } else {
      len = half;
    }
  }
  size_t r = first - 1, hi = size - 2;
  return r > hi ? hi : r;
}
PT_DEV float dist1d_sample(const float* func, const float* cdf, float func_int, int n, float u, float* pdf, size_t* off, const uint32_t* guide,
                           uint32_t K) {  // sampling.rs:164-182
  size_t offset = guide ? find_interval_guided(cdf, (size_t)n + 1, u, guide, K, func) : find_interval_cdf(cdf, (size_t)n + 1, u);
  *off = offset;
  float c0 = __ldg(cdf + offset), c1 = __ldg(cdf + offset + 1);
  float du = u - c0;
  if ((c1 - c0) > 0.0f) du /= c1 - c0;
  *pdf = func_int > 0.0f ? __ldg(func + offset) / func_int : 0.0f;
  return ((float)offset + du) / (float)n;
}
PT_DEV V2 dist2d_sample(const DevEnv& e, V2 u, float* pdf) {  // sampling.rs:211-221
  float p0, p1;
  size_t v, dummy;
  float d1 = dist1d_sample(e.marg_func, e.marg_cdf, e.marg_func_int, e.nv, u.y, &p1, &v, e.marg_guide, e.kv);
  float d0 = dist1d_sample(e.cond_func + v * e.nu, e.cond_cdf + v * (e.nu + 1), __ldg(e.cond_func_int + v), e.nu, u.x, &p0, &dummy,
                           e.cond_guide ? e.cond_guide + v * (e.ku + 1) : nullptr, e.ku);
  *pdf = p0 * p1;
  return V2{d0, d1};
}
PT_DEV float dist2d_pdf(const DevEnv& e, float px, float py) {  // sampling.rs:223-229
  unsigned long long iu = (unsigned long long)(px * (float)e.nu), iv = (unsigned long long)(py * (float)e.nv);
  if (iu > (unsigned long long)e.nu - 1) iu = e.nu - 1;
  if (iv > (unsigned long long)e.nv - 1) iv = e.nv - 1;
  return __ldg(e.cond_func + iv * e.nu + iu) / e.marg_func_int;
}
PT_DEV Spec env_lookup(const DevScene& sc, const DevEnv& e, float s, float t) { return mip_lookup_width(sc, sc.mipmaps[e.mip], s, t, 0.0f); }
// InfiniteAreaLight::le, light.rs:488-498
PT_DEV Spec env_le(const DevScene& sc, const PtrsLight& l, V3 ray_d) {
  const DevEnv& e = sc.envs[l.env];
  V3 w = normalize(xform_vec(e.world_to_light, ray_d));
  return env_lookup(sc, e, spherical_phi(w) * PT_INV_2_PI, spherical_theta(w) * PT_FRAC_1_PI);
}
// DiffuseAreaLight::l at a reconstructed hit (light.rs:252-258 via interaction.rs:297-303)
PT_DEV Spec area_le(const DevScene& sc, int light_id, const SurfInter& si, V3 w) {
  if (light_id < 0) return sp(0.0f);
  if (!(dot(si.g.n, w) > 0.0f)) return sp(0.0f);
  return tex_spec(sc, sc.lights[light_id].ke_tex, tc_of(si));
}

struct TriPoint {  // what Triangle::sample returns that the path reads
  Inter it;
  V2 uv;
};
PT_DEVN TriPoint triangle_sample(const DevScene& sc, int prim, V2 u) {  // shape.rs:541-578
  float su0 = sqrtf(u.x);
  float b0 = 1.0f - su0, b1 = u.y * su0;
  const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim), v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1),
               v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
  const V3 p0 = mk3(v0), p1 = mk3(v1), p2 = mk3(v2);
  const uint32_t flags = __float_as_uint(v2.w) & 0xffu;
  const uint4 idx = __ldg(sc.tri_index + prim);
  TriPoint tp;
  const float b2 = 1.0f - b0 - b1;
  tp.it.p = (b0 * p0) + (b1 * p1) + b2 * p2;
  tp.it.n = normalize(cross(p1 - p0, p2 - p0));
  if (flags & PTRS_MESH_HAS_NORMAL) {
    V3 ns = (b0 * load3(sc.normal, idx.x)) + (b1 * load3(sc.normal, idx.y)) + b2 * load3(sc.normal, idx.z);
    tp.it.n = face_forward(tp.it.n, ns);
  }
  V3 p_abs_sum = vabs(b0 * p0) + vabs(b1 * p1) + vabs(b2 * p2);
  tp.it.p_error = gamma_n(6) * p_abs_sum;
  V2 uv[3];
  tri_uvs(sc, idx, flags, uv);
  tp.uv = V2{b0 * uv[0].x + b1 * uv[1].x + b2 * uv[2].x, b0 * uv[0].y + b1 * uv[1].y + b2 * uv[2].y};
  return tp;
}

// Triangle::pdf_at_point, shape.rs:62-72: a single-triangle Triangle::intersect from `ref` along wi
PT_DEVN float triangle_pdf_at_point(const DevScene& sc, int prim, Inter ref, V3 wi, float area) {
  V3 o;
  spawn_ray(ref, wi, &o);
  const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim), v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1),
               v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
  const V3 p0 = mk3(v0), p1 = mk3(v1), p2 = mk3(v2);
  const RayPre rp = ray_precompute(wi);
  float t, b0, b1, b2;
  if (!tri_core(p0, p1, p2, o, rp, CUDART_INF_F, &t, &b0, &b1, &b2)) return 0.0f;
  if (tri_post_reject(sc, prim, p0, p1, p2, __float_as_uint(v2.w), b0, b1, b2, true)) return 0.0f;
  // isect_light.general.{p, n} of the hit.  On a mesh with normals or tangents the reference's n is the geometric
  // normal flipped towards the shading normal (set_shading_geometry, interaction.rs:194-214) — +-n; only
  // |dot(n, -wi)| is used and negation is exact, so the shading frame of the light's triangle is not rebuilt.
  V3 p_hit = b0 * p0 + b1 * p1 + b2 * p2;
  V3 n = normalize(cross(p0 - p2, p1 - p2));
  return norm_squared(ref.p - p_hit) / (fabsf(dot(n, -wi)) * area);
}


// Light::sample_li (light.rs:97-116 point, :176-196 directional, :262-280 area, :402-441 infinite): incident
// direction, pdf, the far end of the visibility segment and the unoccluded radiance.  pdf == 0 with black Li is what
// the infinite light's early return (map_pdf == 0, where the reference's caller would panic on the missing
// VisibilityTester, integrator.rs:51) becomes here.
struct LightSample {
  V3 wi;
  float pdf;
  Inter p1;  // VisibilityTester.p1
  Spec li;
};
PT_DEV bool light_is_delta(const PtrsLight& light) { return light.type == PTRS_LIGHT_POINT || light.type == PTRS_LIGHT_DIRECTIONAL; }
PT_DEV void light_sample_li(const DevScene& sc, const PtrsLight& light, const Inter& ref, V2 u, LightSample* out) {
  out->wi = mk3(0, 0, 0);
  out->pdf = 0.0f;
  out->p1.p = mk3(0, 0, 0);
  out->p1.p_error = mk3(0, 0, 0);
  out->p1.n = mk3(0, 0, 0);
  out->li = sp(0.f);
  if (light.type == PTRS_LIGHT_POINT) {
    V3 pl = mk3(light.pos[0], light.pos[1], light.pos[2]);
    out->wi = normalize(pl - ref.p);
    out->pdf = 1.0f;
    out->p1.p = pl;
    out->li = sp(light.color[0], light.color[1], light.color[2]) / norm_squared(pl - ref.p);
  } else if (light.type == PTRS_LIGHT_DIRECTIONAL) {
    V3 wl = mk3(light.pos[0], light.pos[1], light.pos[2]);
    out->wi = wl;
    out->pdf = 1.0f;
    out->p1.p = ref.p + wl * (2.0f * light.world_radius);
    out->li = sp(light.color[0], light.color[1], light.color[2]);
  } else if (light.type == PTRS_LIGHT_AREA) {
    TriPoint tp = triangle_sample(sc, light.prim, u);
    out->wi = normalize(tp.it.p - ref.p);
    out->pdf = triangle_pdf_at_point(sc, light.prim, ref, out->wi, light.area);
    out->p1 = tp.it;
    if (dot(tp.it.n, -out->wi) > 0.0f) out->li = tex_spec(sc, light.ke_tex, TexCoord{tp.uv.x, tp.uv.y, 0.f, 0.f, 0.f, 0.f});
  } else {  // PTRS_LIGHT_INFINITE
    const DevEnv& e = sc.envs[light.env];
    float map_pdf = 0.0f;
    V2 uv = dist2d_sample(e, u, &map_pdf);
    if (map_pdf != 0.0f) {
      float theta = uv.y * PT_PI, phi = uv.x * 2.0f * PT_PI;
      float cos_t = cos_small_angle(theta), sin_t = sin_small_angle(theta);
      float sin_p = sin_small_angle(phi), cos_p = cos_small_angle(phi);
      out->wi = xform_vec(e.light_to_world, mk3(sin_t * cos_p, sin_t * sin_p, cos_t));
      out->pdf = sin_t == 0.0f ? 0.0f : map_pdf / (2.0f * PT_PI * PT_PI * sin_t);
      out->p1.p = ref.p + out->wi * (2.0f * light.world_radius);
      out->li = env_lookup(sc, e, uv.x, uv.y);
    }
  }
}
// Light::pdf_li for the lights that have one (area light.rs:286-288, infinite :447-461; delta lights return 0)
PT_DEV float light_pdf_li(const DevScene& sc, const PtrsLight& light, const Inter& ref, V3 w) {
  if (light.type == PTRS_LIGHT_AREA) return triangle_pdf_at_point(sc, light.prim, ref, w, light.area);
  if (light.type != PTRS_LIGHT_INFINITE) return 0.0f;
  const DevEnv& e = sc.envs[light.env];
  V3 wl = xform_vec(e.world_to_light, w);
  float theta = spherical_theta(wl), phi = spherical_phi(wl);
  float sin_t = sin_small_angle(theta);
  return sin_t == 0.0f ? 0.0f : dist2d_pdf(e, phi * PT_INV_2_PI, theta * PT_FRAC_1_PI) / (2.0f * PT_PI * PT_PI * sin_t);
}

}  // namespace ptrs
