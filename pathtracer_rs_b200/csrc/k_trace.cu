// extend / connect / standalone intersect kernels (BVH traversal lives only in this unit)
#include "launch.hpp"
#include "wavefront.cuh"

#define PT_TRACE_MIN_BLOCKS 8

namespace ptrs {

// Opportunistic warp aggregation for queue appends issued from divergent code: the lanes that are
// converged here and target the same counter share one atomicAdd.
PT_DEV uint32_t coalesced_slot(uint32_t* counter) {
  const uint32_t m = __activemask();
  const uint32_t grp = __match_any_sync(m, (unsigned long long)(uintptr_t)counter);
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(grp) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(grp));
  base = __shfl_sync(grp, base, leader);
  return base + (uint32_t)__popc(grp & ((1u << lane) - 1u));
}

// ---- extend ----------------------------------------------------------------------------------------
// Closest hit for every path of the round's extend queue (integrator.rs:416); the hit's material type
// picks the shade queue the path is appended to (material sorting).
struct ExtendWork {
  const DevScene& sc;
  const PathArrays& P;
  const int* __restrict__ q_ext;
  int* __restrict__ q_class;
  uint32_t cap;
  RoundCounters* ctr;
  int p;
  __device__ bool begin(uint32_t i, LaneRay* r) {
    p = q_ext[i];
    const PathRay pr = ld256(&P.slot[p].r);
    r->o = mk3(pr.ox, pr.oy, pr.oz);
    r->d = mk3(pr.dx, pr.dy, pr.dz);
    r->t_max = CUDART_INF_F;
    r->any_hit = false;
    return true;
  }
  __device__ bool end(uint32_t, const DevHit& h, bool found, LaneRay*) {
    const int cls = found ? sc.materials[__float_as_int(__ldg(&sc.tri_verts[3 * (size_t)h.prim].w))].type : PT_CLASS_MISS;
    const size_t slot = (size_t)cls * cap + coalesced_slot(&ctr->n_class[cls]);
    q_class[slot] = p;
    if (found) P.q_hit[slot] = make_float4(__int_as_float(h.prim), h.b0, h.b1, h.b2);
    return false;
  }
};

template <bool COUNT, bool DIST>
__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) extend_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ PathArrays P, const int* __restrict__ q_ext, int* __restrict__ q_class,
                                                      uint32_t cap, RoundCounters* ctr, GlobalCounters* g) {
  uint32_t c_nodes = 0, c_tris = 0;
  ExtendWork w{sc, P, q_ext, q_class, cap, ctr, 0};
  trace_stream<COUNT, DIST>(sc, ctr->n_ext, &ctr->t_ext, w, &c_nodes, &c_tris);
  if (COUNT) {
    warp_sum_add(c_nodes, &g->nodes_tested);
    warp_sum_add(c_tris, &g->tris_tested);
  }
}

// ---- connect ---------------------------------------------------------------------------------------
// Rays of estimate_direct for the pending records: shade lists in q_ray the rays that exist, 2 * record for a
// shadow segment (integrator.rs:66-78, light.rs:39-41, any-hit), 2 * record + 1 for a BSDF-sampled MIS ray
// (integrator.rs:113-135, closest hit), so every work item is a ray and no lane idles on an absent one.  Any-hit rays sit
// at the bottom of q_ray (n_ray of them), closest-hit ones at the top (n_ray_closest): work item i < n_low is q_ray[i],
// the rest count down from q_ray[2 * cap - 1].  The kernel only traces: what was found goes to nee_res[i], and connect_resolve_kernel
// (k_misc.cu) evaluates emitted radiance and adds the bounce's direct lighting at full warp width.
struct ConnectWork {
  const PathArrays& P;
  uint32_t n_low, top;  // top = 2 * cap - 1
  uint32_t n_shadow, n_mis;
  uint32_t cur;  // 2 * record + kind of the ray in hand
  __device__ bool begin(uint32_t i, LaneRay* r) {
    cur = P.q_ray[i < n_low ? i : top - (i - n_low)];
    const uint32_t rec = cur >> 1;
    if (cur & 1u) {
      const F8 n23 = ld256(reinterpret_cast<const F8*>(&P.nee[rec].n2));
      r->o = mk3(n23.a);
      r->d = mk3(n23.b);
      r->t_max = CUDART_INF_F;
      r->any_hit = (__float_as_uint(n23.b.w) & PT_NEE_MIS_ANY) != 0;  // infinite light: only "does it escape" matters
      ++n_mis;
    } else {
      const F8 n01 = ld256(reinterpret_cast<const F8*>(&P.nee[rec].n0));
      r->o = mk3(n01.a);
      r->d = mk3(n01.b);
      r->t_max = 1.0f - PT_SHADOW_EPSILON;
      r->any_hit = true;
      ++n_shadow;
    }
    return true;
  }
  __device__ bool end(uint32_t, const DevHit& h, bool found, LaneRay*) {
    NeeRes* res = P.nee_res + (cur >> 1);
    if (cur & 1u) *reinterpret_cast<float4*>(res) = make_float4(__int_as_float(found ? h.prim : -1), h.b0, h.b1, h.b2);
    else res->occluded = found ? 1u : 0u;
    return false;
  }
};

// every ray of the round, or (closest_only) the closest-hit MIS rays when occlusion_kernel has traced the any-hit ones
template <bool COUNT, bool DIST>
__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) connect_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ PathArrays P, uint32_t cap,
                                                                           bool closest_only, RoundCounters* ctr, GlobalCounters* g) {
  uint32_t c_nodes = 0, c_tris = 0;
  const uint32_t n_low = closest_only ? 0u : ctr->n_ray;
  ConnectWork w{P, n_low, 2u * cap - 1u, 0u, 0u, 0u};
  trace_stream<COUNT, DIST>(sc, n_low + ctr->n_ray_closest, closest_only ? &ctr->t_ray_closest : &ctr->t_ray, w, &c_nodes, &c_tris);
  warp_sum_add(w.n_shadow, &g->shadow_rays);
  warp_sum_add(w.n_mis, &g->mis_rays);
  if (COUNT) {
    warp_sum_add(c_nodes, &g->nee_nodes_tested);
    warp_sum_add(c_tris, &g->nee_tris_tested);
  }
}

// the any-hit rays of the round over the occlusion tree
__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) occlusion_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ PathArrays P, RoundCounters* ctr, GlobalCounters* g) {
  const uint32_t n = ctr->n_ray;
  ConnectWork w{P, n, 0u, 0u, 0u, 0u};
  trace_occlusion(sc, n, &ctr->t_ray, w);
  warp_sum_add(w.n_shadow, &g->shadow_rays);
  warp_sum_add(w.n_mis, &g->mis_rays);
}

// ---- standalone traversal kernels (ptrs_intersect*, the BVH microbenchmark) --------------------------
struct IntersectWork {
  const PtrsRay* __restrict__ rays;
  PtrsHit* __restrict__ hits;
  uint8_t* __restrict__ occluded;
  bool any_hit;
  const uint32_t* __restrict__ prim_map;  // BVH position -> caller's primitive index (device-built BVH), or null
  __device__ bool begin(uint32_t i, LaneRay* r) {
    const float* q = (const float*)(rays + i);
    r->o = mk3(__ldg(q), __ldg(q + 1), __ldg(q + 2));
    r->d = mk3(__ldg(q + 3), __ldg(q + 4), __ldg(q + 5));
    r->t_max = __ldg(q + 6);
    r->any_hit = any_hit;
    return true;
  }
  __device__ bool end(uint32_t i, const DevHit& h, bool found, LaneRay*) {
    if (any_hit) {
      occluded[i] = found ? 1 : 0;
    } else {
      PtrsHit out;
      out.prim = found ? (prim_map ? (int)__ldg(prim_map + h.prim) : h.prim) : -1;
      out.t = found ? h.t : 0.f;
      out.b0 = h.b0;
      out.b1 = h.b1;
      out.b2 = h.b2;
      hits[i] = out;
    }
    return false;
  }
};

template <bool ANY_HIT, bool COUNT, bool DIST>
__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) intersect_kernel(const __grid_constant__ DevScene sc, const PtrsRay* __restrict__ rays, uint32_t n, PtrsHit* __restrict__ hits,
                                                         uint8_t* __restrict__ occluded, uint32_t* ticket, GlobalCounters* g, const uint32_t* __restrict__ prim_map) {
  uint32_t c_nodes = 0, c_tris = 0;
  IntersectWork w{rays, hits, occluded, ANY_HIT, prim_map};
  trace_stream<COUNT, DIST>(sc, n, ticket, w, &c_nodes, &c_tris);
  if (COUNT) {
    warp_sum_add(c_nodes, &g->nodes_tested);
    warp_sum_add(c_tris, &g->tris_tested);
  }
}

__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) intersect_p_occlusion_kernel(const __grid_constant__ DevScene sc, const PtrsRay* __restrict__ rays, uint32_t n,
                                                                                         uint8_t* __restrict__ occluded, uint32_t* ticket) {
  IntersectWork w{rays, nullptr, occluded, true, nullptr};
  trace_occlusion(sc, n, ticket, w);
}

// ---- launchers -----------------------------------------------------------------------------------------
// <.., DIST>: front-to-back child order on trees the library built (DevScene::dist_order); the counted variants read the flag at
// run time, so they exist once
void launch_extend(cudaStream_t st, int sm, bool count, const DevScene& sc, const PathArrays& P, const int* q_ext, int* q_class, uint32_t cap,
                   RoundCounters* ctr, GlobalCounters* g) {
  if (count) extend_kernel<true, false><<<PT_GRID((extend_kernel<true, false>), 128, sm), 128, 0, st>>>(sc, P, q_ext, q_class, cap, ctr, g);
  else if (sc.dist_order) extend_kernel<false, true><<<PT_GRID((extend_kernel<false, true>), 128, sm), 128, 0, st>>>(sc, P, q_ext, q_class, cap, ctr, g);
  else extend_kernel<false, false><<<PT_GRID((extend_kernel<false, false>), 128, sm), 128, 0, st>>>(sc, P, q_ext, q_class, cap, ctr, g);
}
void launch_connect(cudaStream_t st, int sm, bool count, const DevScene& sc, const PathArrays& P, uint32_t cap, bool closest_only, RoundCounters* ctr,
                    GlobalCounters* g) {
  if (count) connect_kernel<true, false><<<PT_GRID((connect_kernel<true, false>), 128, sm), 128, 0, st>>>(sc, P, cap, closest_only, ctr, g);
  else if (sc.dist_order) connect_kernel<false, true><<<PT_GRID((connect_kernel<false, true>), 128, sm), 128, 0, st>>>(sc, P, cap, closest_only, ctr, g);
  else connect_kernel<false, false><<<PT_GRID((connect_kernel<false, false>), 128, sm), 128, 0, st>>>(sc, P, cap, closest_only, ctr, g);
}
void launch_occlusion(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, RoundCounters* ctr, GlobalCounters* g) {
  occlusion_kernel<<<PT_GRID(occlusion_kernel, 128, sm), 128, 0, st>>>(sc, P, ctr, g);
}
void launch_intersect(cudaStream_t st, int sm, bool any_hit, bool count, const DevScene& sc, const PtrsRay* rays, uint32_t n, PtrsHit* hits,
                      uint8_t* occluded, uint32_t* ticket, GlobalCounters* g, const uint32_t* prim_map) {
#define PT_LAUNCH_INTERSECT(A, C, D) \
  intersect_kernel<A, C, D><<<PT_GRID((intersect_kernel<A, C, D>), 128, sm), 128, 0, st>>>(sc, rays, n, hits, occluded, ticket, g, prim_map)
  const bool dist = sc.dist_order != 0;
  if (any_hit && !count && sc.n_wnodes > 0) intersect_p_occlusion_kernel<<<PT_GRID(intersect_p_occlusion_kernel, 128, sm), 128, 0, st>>>(sc, rays, n, occluded, ticket);
  else if (!any_hit && count) PT_LAUNCH_INTERSECT(false, true, false);
  else if (any_hit && count) PT_LAUNCH_INTERSECT(true, true, false);
  else if (!any_hit && dist) PT_LAUNCH_INTERSECT(false, false, true);
  else if (!any_hit) PT_LAUNCH_INTERSECT(false, false, false);
  else if (dist) PT_LAUNCH_INTERSECT(true, false, true);
  else PT_LAUNCH_INTERSECT(true, false, false);
#undef PT_LAUNCH_INTERSECT
}

}  // namespace ptrs
