// shade<MAT> kernel; compiled once per material type with -DPT_SHADE_MAT=<n> so the six
// instantiations build in parallel and each gets its own register allocation
#include "launch.hpp"
#include "wavefront.cuh"

namespace ptrs {

// first half of estimate_direct (integrator.rs:38-80): light sample, BSDF eval, shadow segment; and
// the BSDF-sampling half up to the point where a ray must be traced (integrator.rs:82-114)
PT_DEV void nee_prepare(const DevScene& sc, const SurfInter& si, const Bsdf& bsdf, V2 u_scattering, int light_idx, V2 u_light,
                        float4* n0, float4* n1, float4* n2, float4* n3, float4* n4, float* scat_pdf_out, uint32_t* nee_flags) {
  const PtrsLight& light = sc.lights[light_idx];
  const uint32_t bsdf_flags = BSDF_ALL & ~BSDF_SPECULAR;
  float scattering_pdf = 0.0f;
  const bool delta = light_is_delta(light);
  LightSample ls;
  light_sample_li(sc, light, si.g, u_light, &ls);
  const V3 wi = ls.wi;
  const float light_pdf = ls.pdf;
  const Inter& p1 = ls.p1;
  const Spec li = ls.li;
  uint32_t nf = (uint32_t)light_idx;
  Spec A = sp(0.f);
  V3 sh_o = mk3(0, 0, 0), sh_d = mk3(0, 0, 0);
  if (light_pdf > 0.0f && !is_black(li)) {
    Spec f = bsdf_f(bsdf, si.wo, wi, bsdf_flags) * fabsf(dot(wi, si.sh_n));
    scattering_pdf = bsdf_pdf(bsdf, si.wo, wi, bsdf_flags);
    if (!is_black(f)) {
      spawn_ray_to_it(si.g, p1, &sh_o, &sh_d);
      nf |= PT_NEE_SHADOW;
      if (delta) A = f * li / light_pdf;
      else A = f * li * power_heuristic(light_pdf, scattering_pdf) / light_pdf;
    }
  }
  V3 mo = mk3(0, 0, 0), md = mk3(0, 0, 0);
  Spec f2 = sp(0.f);
  float weight = 1.0f;
  if (!delta) {
    uint32_t sampled_type = BSDF_ALL;
    V3 wi2 = mk3(0, 0, 0);
    f2 = bsdf_sample_f(bsdf, si.wo, &wi2, u_scattering, &scattering_pdf, bsdf_flags, &sampled_type);
    f2 = f2 * fabsf(dot(wi2, si.sh_n));
    const bool sampled_specular = (sampled_type & BSDF_SPECULAR) == BSDF_SPECULAR;
    if (!is_black(f2) && scattering_pdf > 0.0f) {
      bool go = true;
      if (!sampled_specular) {
        const float lp = light_pdf_li(sc, light, si.g, wi2);
        if (lp == 0.0f) go = false;  // `return ld` (integrator.rs:107-109)
        else weight = power_heuristic(scattering_pdf, lp);
      }
      if (go) {
        spawn_ray(si.g, wi2, &mo);
        md = wi2;
        nf |= PT_NEE_MIS | (light.type == PTRS_LIGHT_INFINITE ? PT_NEE_MIS_ANY : 0u);
      }
    }
  }
  *n0 = make_float4(sh_o.x, sh_o.y, sh_o.z, A.r);
  *n1 = make_float4(sh_d.x, sh_d.y, sh_d.z, A.g);
  *n2 = make_float4(mo.x, mo.y, mo.z, A.b);
  *n3 = make_float4(md.x, md.y, md.z, __uint_as_float(nf));
  *n4 = make_float4(f2.r, f2.g, f2.b, weight);
  *scat_pdf_out = scattering_pdf;
  *nee_flags = nf;
}

#ifndef PT_SHADE_PARAM
#define PT_SHADE_PARAM  // by value: with __grid_constant__ the 128-register shade kernels spill more (measured slower)
#endif
#ifndef PT_SHADE_MIN_BLOCKS
#define PT_SHADE_MIN_BLOCKS 4
#endif
#ifndef PT_SHADE_BLOCK
#define PT_SHADE_BLOCK 128
#endif

// EXACT only names the build: the exact instantiation comes from a translation unit compiled with IEEE division /
// square root and without FMA contraction (PtrsRenderParams.flags & PTRS_RENDER_EXACT_SHADING, Makefile EXACTSHADE),
// the other from the fast-math-free but contracted default build; the source is the same.
#ifndef PT_SHADE_EXACT
#define PT_SHADE_EXACT 0
#endif
template <int MAT, bool EXACT>
__global__ void __launch_bounds__(PT_SHADE_BLOCK, PT_SHADE_MIN_BLOCKS) shade_kernel(const __grid_constant__ RenderConst rc, PT_SHADE_PARAM DevScene sc, PT_SHADE_PARAM PathArrays P,
                                                     const int* __restrict__ q, const float4* __restrict__ q_hit, int* __restrict__ q_ext_next,
                                                     int* __restrict__ q_nee, RoundCounters* ctr, RoundCounters* ctr_next) {
  const uint32_t n = ctr->n_class[MAT];
  const int lane = threadIdx.x & 31;
  const uint32_t* __restrict__ sobol = sc.sobol;
  // shade work is uniform per item (one material type per launch): static striding, no ticket atomic
  const uint32_t warp_stride = (gridDim.x * blockDim.x) & ~31u;
  uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u;
  // the item after this one is known one iteration ahead: its slot record and triangle are prefetched while
  // the current item is shaded
  int p_next = 0, prim_next = 0;
  if (base + lane < n) {
    p_next = q[base + lane];
    prim_next = __float_as_int(q_hit[base + lane].x);
  }
  for (; base < n; base += warp_stride) {
    const uint32_t i = base + lane;
    bool push_ext = false, push_nee = false;
    const int p = p_next;
    NeeRec nee;
    if (i < n) {
      const int prim = prim_next;
      const float4 hb = q_hit[i];
      const PathRay pr = ld256(&P.slot[p].r);
      const PathAux pa = ld256(&P.slot[p].a);
      const uint32_t i_next = i + warp_stride;
      if (i_next < n) {
        p_next = q[i_next];
        prim_next = __float_as_int(q_hit[i_next].x);
      }
      const V3 ray_d = mk3(pr.dx, pr.dy, pr.dz);
      SurfInter si;
      reconstruct_hit(sc, prim, hb.y, hb.z, hb.w, ray_d, &si);
      if (i_next < n) {
        prefetch_l1(&P.slot[p_next]);
        prefetch_l1(sc.tri_verts + 3 * (size_t)prim_next);
        prefetch_l1(sc.tri_verts + 3 * (size_t)prim_next + 2);
#if PT_PACKED_SHADING
        prefetch_l1(sc.tri_shade + 4 * (size_t)prim_next);
#else
        prefetch_l1(sc.tri_index + prim_next);
#endif
      }
      uint32_t flags = pr.packed & 0x00ffffffu;
      int bounces = packed_bounces(pr.packed);
      Spec beta = sp(pa.br, pa.bg, pa.bb);
      float eta_scale = pr.eta_scale;
      const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim), v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1);
      const int mat_id = __float_as_int(v0.w), light_id = __float_as_int(v1.w);
      // emitted radiance at the vertex (integrator.rs:418-422)
      if (bounces == 0 || (flags & PT_F_SPECULAR)) {
        const Spec add = beta * area_le(sc, light_id, si, -ray_d);
        if (!is_black(add)) {  // L + 0 == L: the read-modify-write is skipped for the (common) non-emitter
          const float4 l4 = P.L[p];
          const Spec L = sp(l4.x, l4.y, l4.z) + add;
          P.L[p] = make_float4(L.r, L.g, L.b, 0.f);
        }
      }
      bool alive = bounces < rc.max_depth;  // integrator.rs:429
      if (alive) {
        if ((flags & PT_F_HAS_DIFF) && sc.uses_differentials) {  // compute_scattering_functions -> compute_differentials
          RayDiff rd;
          V3 o, d;
          camera_ray(rc.cam, pa.fx, pa.fy, rc.diff_scale, &o, &d, &rd.rx_d, &rd.ry_d);
          rd.rx_o = o;
          rd.ry_o = o;
          compute_differentials(&si, rd);
        }
        flags &= ~PT_F_HAS_DIFF;
        const PtrsMaterial& m = sc.materials[mat_id];
        Bsdf bsdf;
        PathRay out = pr;
        bool do_nee = false;
        V2 u_light = V2{0.f, 0.f}, u_scattering = V2{0.f, 0.f};
        float u_idx = 0.f;
        const Spec beta0 = beta;  // throughput before this bounce: what the direct-lighting estimate is weighted by
        if (!compute_scattering_functions<MAT>(sc, m, &si, &bsdf)) {
          // null BSDF: continue straight through; `bounces -= 1; continue` nets -1 (integrator.rs:434-439)
          V3 o;
          spawn_ray(si.g, ray_d, &o);
          out.ox = o.x;
          out.oy = o.y;
          out.oz = o.z;
          bounces -= 1;
          push_ext = true;
        } else {
          PathSampler ps;
          const int2 pix = unpack_pixel(pa.pixel);
          sampler_start(rc.sobol, rc.split, ps, pix.x, pix.y, pa.sample, flags & 0xffffu);
          // direct lighting (integrator.rs:443-447, 192-217): its five sample values are drawn here, in the
          // reference's order; the estimate itself runs after the path's continuation has been stored, when the
          // path state is dead and before the 96-byte record becomes live
          if (bsdf_num_components(bsdf, BSDF_ALL & ~BSDF_SPECULAR) > 0 && sc.n_lights > 0) {
            do_nee = true;
            u_light = get_2d(rc.sobol, rc.split, sobol, ps);
            u_scattering = get_2d(rc.sobol, rc.split, sobol, ps);
            u_idx = get_1d(rc.sobol, rc.split, sobol, ps);
          }
          // continuation (integrator.rs:449-499)
          V3 wi = mk3(0, 0, 0);
          float pdf = 0.0f;
          uint32_t sampled = 0;
          Spec f = bsdf_sample_f(bsdf, si.wo, &wi, get_2d(rc.sobol, rc.split, sobol, ps), &pdf, BSDF_ALL, &sampled);
          if (!(is_black(f) || pdf == 0.0f)) {
            beta = beta * (f * fabsf(dot(wi, si.sh_n)) / pdf);
            if (sampled & BSDF_SPECULAR) flags |= PT_F_SPECULAR;
            else flags &= ~PT_F_SPECULAR;
            if ((sampled & BSDF_SPECULAR) && (sampled & BSDF_TRANSMISSION)) {
              float eta = bsdf.eta;
              eta_scale *= dot(si.wo, si.g.n) > 0.0f ? eta * eta : 1.0f / (eta * eta);
            }
            V3 o;
            spawn_ray(si.g, wi, &o);
            bool survive = true;
            if (rc.rr_enable) {
              Spec rr_beta = beta * eta_scale;
              float mc = max_component(rr_beta);
              if (mc < rc.rr_threshold && bounces > rc.rr_start_depth) {
                float qv = fmaxf(0.05f, 1.0f - mc);
                if (get_1d(rc.sobol, rc.split, sobol, ps) < qv) survive = false;
                else beta = beta / (1.0f - qv);
              }
            }
            if (survive) {
              out.ox = o.x;
              out.oy = o.y;
              out.oz = o.z;
              out.dx = wi.x;
              out.dy = wi.y;
              out.dz = wi.z;
              bounces += 1;
              push_ext = true;
            }
          }
          flags = (flags & 0xffff0000u) | (ps.dimension & 0xffffu);
        }
        if (push_ext) {
          out.packed = pack_state(flags, bounces);
          out.eta_scale = eta_scale;
          PathAux oa = pa;
          oa.br = beta.r;
          oa.bg = beta.g;
          oa.bb = beta.b;
          st256(&P.slot[p].r, out);
          st256(&P.slot[p].a, oa);
        }
        if (do_nee) {
          unsigned long long li64 = (unsigned long long)floorf(u_idx * (float)sc.n_lights);
          int light_idx = (int)(li64 < (unsigned long long)(sc.n_lights - 1) ? li64 : (unsigned long long)(sc.n_lights - 1));
          float scat_pdf;
          uint32_t nf;
          nee_prepare(sc, si, bsdf, u_scattering, light_idx, u_light, &nee.n0, &nee.n1, &nee.n2, &nee.n3, &nee.n4, &scat_pdf, &nf);
          if (nf & (PT_NEE_SHADOW | PT_NEE_MIS)) {
            nee.n5 = make_float4(beta0.r, beta0.g, beta0.b, scat_pdf);
            push_nee = true;
          }
        }
      }
    }
    // the appends of the warp (connect queue with its 96-byte record, the rays of those records, next extend
    // queue): one atomic each, in flight together
    {
      const uint32_t nfl = push_nee ? __float_as_uint(nee.n3.w) : 0u;
      const uint32_t ma = __ballot_sync(0xffffffffu, push_nee), mb = __ballot_sync(0xffffffffu, push_ext);
      // any-hit rays (shadow segments, MIS rays of infinite lights) fill q_ray from the bottom, closest-hit MIS rays (area
      // lights) from the top down: connect traces the two lists with different kernels
      const uint32_t ms = __ballot_sync(0xffffffffu, (nfl & PT_NEE_SHADOW) != 0);
      const uint32_t mm = __ballot_sync(0xffffffffu, (nfl & (PT_NEE_MIS | PT_NEE_MIS_ANY)) == (PT_NEE_MIS | PT_NEE_MIS_ANY));
      const uint32_t mc = __ballot_sync(0xffffffffu, (nfl & (PT_NEE_MIS | PT_NEE_MIS_ANY)) == PT_NEE_MIS);
      uint32_t ba = 0, bb = 0, br = 0, bc = 0;
      if (lane == 0) {
        if (ma) {
          const unsigned long long both = atomicAdd(reinterpret_cast<unsigned long long*>(&ctr->n_nee),
                                                    (unsigned long long)__popc(ma) | ((unsigned long long)(__popc(ms) + __popc(mm)) << 32));
          ba = (uint32_t)both;
          br = (uint32_t)(both >> 32);
        }
        if (mc) bc = atomicAdd(&ctr->n_ray_closest, (uint32_t)__popc(mc));
        if (mb) bb = atomicAdd(&ctr_next->n_ext, (uint32_t)__popc(mb));
      }
      ba = __shfl_sync(0xffffffffu, ba, 0);
      bb = __shfl_sync(0xffffffffu, bb, 0);
      br = __shfl_sync(0xffffffffu, br, 0);
      bc = __shfl_sync(0xffffffffu, bc, 0);
      const uint32_t lt = (1u << lane) - 1u;
      if (push_nee) {
        const uint32_t k = ba + __popc(ma & lt);
        q_nee[k] = p;
        F8* dst = reinterpret_cast<F8*>(&P.nee[k]);
        st256(dst, F8{nee.n0, nee.n1});
        st256(dst + 1, F8{nee.n2, nee.n3});
        st256(dst + 2, F8{nee.n4, nee.n5});
        if (nfl & PT_NEE_SHADOW) P.q_ray[br + __popc(ms & lt)] = 2u * k;
        if ((mm >> lane) & 1u) P.q_ray[br + __popc(ms) + __popc(mm & lt)] = 2u * k + 1u;
        if ((mc >> lane) & 1u) P.q_ray[2u * rc.cap - 1u - (bc + __popc(mc & lt))] = 2u * k + 1u;
      }
      if (push_ext) q_ext_next[bb + __popc(mb & lt)] = p;
    }
  }
}


// ---- launcher ------------------------------------------------------------------------------------------
#ifndef PT_SHADE_MAT
#error "compile k_shade.cu with -DPT_SHADE_MAT=<PtrsMaterialType>"
#endif
#define PT_CAT2(a, b) a##b
#define PT_CAT(a, b) PT_CAT2(a, b)
#if PT_SHADE_EXACT
#define PT_SHADE_LAUNCHER PT_CAT(launch_shade_exact_, PT_SHADE_MAT)
#else
#define PT_SHADE_LAUNCHER PT_CAT(launch_shade_, PT_SHADE_MAT)
#endif
void PT_SHADE_LAUNCHER(cudaStream_t st, int sm, const RenderConst& rc, const DevScene& sc, const PathArrays& P, const int* q,
                                         const float4* q_hit, int* q_next, int* q_nee, RoundCounters* ctr, RoundCounters* ctr_next) {
  shade_kernel<PT_SHADE_MAT, PT_SHADE_EXACT != 0><<<PT_GRID((shade_kernel<PT_SHADE_MAT, PT_SHADE_EXACT != 0>), PT_SHADE_BLOCK, sm), PT_SHADE_BLOCK, 0, st>>>(rc, sc, P, q, q_hit, q_next, q_nee, ctr, ctr_next);
}

}  // namespace ptrs
