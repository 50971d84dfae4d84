// BVH traversal and watertight ray/triangle intersection on the device.
//   Bounds3::intersect_p_precomp   src/common/bounds.rs:190-232
//   Triangle::intersect(_p)        src/pathtracer/shape.rs:74-185, 362-524
//   BVH::intersect / intersect_p   src/pathtracer/accelerator.rs:359-475
// The visit order (near child first by dir_is_neg[axis], 64-entry stack, triangles of a leaf in
// array order, current t_max used for every later box test) is the reference's, so ties at equal t
// resolve to the same primitive and node / triangle test counts equal the CPU path's.
#pragma once
#include "dev_texture.cuh"

namespace ptrs {

struct RayPre {  // per-ray constants of the triangle test (shape.rs:94-110); kx = kz+1 mod 3, ky = kx+1 mod 3
  int kz;
  float sx, sy, sz;
};
// (v[kx], v[ky], v[kz]) — a cyclic rotation selected by kz
PT_DEV V3 permute(V3 v, int kz) {
  const bool z0 = kz == 0, z1 = kz == 1;
  return mk3(z0 ? v.y : (z1 ? v.z : v.x), z0 ? v.z : (z1 ? v.x : v.y), z0 ? v.x : (z1 ? v.y : v.z));
}

PT_DEV RayPre ray_precompute(V3 d) {
  RayPre p;
  p.kz = max_dimension(vabs(d));
  const V3 dp = permute(d, p.kz);
  p.sx = -dp.x / dp.z;
  p.sy = -dp.y / dp.z;
  p.sz = 1.0f / dp.z;
  return p;
}

// shape.rs:85-185.  Returns true and (t, b0, b1, b2) if the triangle is hit within (0, t_max].
PT_DEV bool tri_core(V3 p0, V3 p1, V3 p2, V3 o, const RayPre& rp, float t_max, float* t_out, float* b0o, float* b1o, float* b2o) {
  const V3 q0 = permute(p0 - o, rp.kz), q1 = permute(p1 - o, rp.kz), q2 = permute(p2 - o, rp.kz);
  float p0x = q0.x, p0y = q0.y, p0z = q0.z;
  float p1x = q1.x, p1y = q1.y, p1z = q1.z;
  float p2x = q2.x, p2y = q2.y, p2z = q2.z;
  p0x += rp.sx * p0z;
  p0y += rp.sy * p0z;
  p1x += rp.sx * p1z;
  p1y += rp.sy * p1z;
  p2x += rp.sx * p2z;
  p2y += rp.sy * p2z;
  float e0 = p1x * p2y - p1y * p2x;
  float e1 = p2x * p0y - p2y * p0x;
  float e2 = p0x * p1y - p0y * p1x;
  if (e0 == 0.0f || e1 == 0.0f || e2 == 0.0f) {
    double p2txp1ty = (double)p2x * (double)p1y, p2typ1tx = (double)p2y * (double)p1x;
    e0 = (float)(p2typ1tx - p2txp1ty);
    double p0txp2ty = (double)p0x * (double)p2y, p0typ2tx = (double)p0y * (double)p2x;
    e1 = (float)(p0typ2tx - p0txp2ty);
    double p1txp0ty = (double)p1x * (double)p0y, p1typ0tx = (double)p1y * (double)p0x;
    e2 = (float)(p1typ0tx - p1txp0ty);
  }
  if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
  float det = e0 + e1 + e2;
  if (det == 0.0f) return false;
  p0z *= rp.sz;
  p1z *= rp.sz;
  p2z *= rp.sz;
  float t_scaled = e0 * p0z + e1 * p1z + e2 * p2z;
  if (det < 0.0f && (t_scaled >= 0.0f || t_scaled < t_max * det)) return false;
  else if (det > 0.0f && (t_scaled <= 0.0f || t_scaled > t_max * det)) return false;
  float inv_det = 1.0f / det;
  float b0 = e0 * inv_det, b1 = e1 * inv_det, b2 = e2 * inv_det;
  float t = t_scaled * inv_det;
  float max_z_t = fmaxf(fmaxf(fabsf(p0z), fabsf(p1z)), fabsf(p2z));
  float delta_z = gamma_n(3) * max_z_t;
  float max_x_t = fmaxf(fmaxf(fabsf(p0x), fabsf(p1x)), fabsf(p2x));
  float max_y_t = fmaxf(fmaxf(fabsf(p0y), fabsf(p1y)), fabsf(p2y));
  float delta_x = gamma_n(5) * (max_x_t + max_z_t);
  float delta_y = gamma_n(5) * (max_y_t + max_z_t);
  float delta_e = 2.0f * (gamma_n(2) * max_x_t * max_y_t + delta_y * max_x_t + delta_x * max_y_t);
  float max_e = fmaxf(fmaxf(fabsf(e0), fabsf(e1)), fabsf(e2));
  float delta_t = 3.0f * (gamma_n(3) * max_e * max_z_t + delta_e * max_z_t + delta_z * max_e) * fabsf(inv_det);
  if (t <= delta_t) return false;
  *t_out = t;
  *b0o = b0;
  *b1o = b1;
  *b2o = b2;
  return true;
}

// default UVs (shape.rs:34-48) or mesh UVs
PT_DEV void tri_uvs(const DevScene& sc, uint4 idx, uint32_t mesh_flags, V2 uv[3]) {
  if (mesh_flags & PTRS_MESH_HAS_UV) {
    const float2* u = (const float2*)sc.uv;
    float2 a = __ldg(u + idx.x), b = __ldg(u + idx.y), c = __ldg(u + idx.z);
    uv[0] = V2{a.x, a.y};
    uv[1] = V2{b.x, b.y};
    uv[2] = V2{c.x, c.y};
  } else {
    uv[0] = V2{0.f, 0.f};
    uv[1] = V2{1.f, 0.f};
    uv[2] = V2{1.f, 1.f};
  }
}

// dpdu / dpdv, shape.rs:187-215; false = degenerate triangle ("the intersection is bogus")
PT_DEV bool tri_partials(V3 p0, V3 p1, V3 p2, const V2 uv[3], V3* dpdu, V3* dpdv) {
  *dpdu = mk3(0, 0, 0);
  *dpdv = mk3(0, 0, 0);
  float duv02x = uv[0].x - uv[2].x, duv02y = uv[0].y - uv[2].y;
  float duv12x = uv[1].x - uv[2].x, duv12y = uv[1].y - uv[2].y;
  V3 dp02 = p0 - p2, dp12 = p1 - p2;
  float determinant = duv02x * duv12y - duv02y * duv12x;
  bool degenerate_uv = fabsf(determinant) < 1e-8f;
  if (!degenerate_uv) {
    float invdet = 1.0f / determinant;
    *dpdu = (duv12y * dp02 - duv02y * dp12) * invdet;
    *dpdv = (-duv12x * dp02 + duv02x * dp12) * invdet;
  }
  if (degenerate_uv || norm_squared(cross(*dpdu, *dpdv)) == 0.0f) {
    V3 ng = cross(p2 - p0, p1 - p0);
    if (norm_squared(ng) == 0.0f) return false;
    coordinate_system(normalize(ng), dpdu, dpdv);
  }
  return true;
}

// The part of Triangle::intersect after the t test that can still reject the hit: degenerate
// partials (shape.rs:205-212) — only reachable for zero-area triangles — and the alpha mask
// (shape.rs:228-244).  Slow path, taken only for primitives whose mesh has an alpha texture or
// for closest-hit candidates (any-hit only evaluates partials under an alpha mask, shape.rs:471).
PT_DEVN bool tri_post_reject_slow(const DevScene& sc, int prim, V3 p0, V3 p1, V3 p2, uint32_t meta2, float b0, float b1, float b2) {
  const bool has_alpha = (meta2 & PT_TRI_ALPHA_BIT) != 0;
  uint4 idx = __ldg(sc.tri_index + prim);
  V2 uv[3];
  tri_uvs(sc, idx, meta2 & 0xffu, uv);
  V3 dpdu, dpdv;
  if (!tri_partials(p0, p1, p2, uv, &dpdu, &dpdv)) return true;
  if (has_alpha) {
    TexCoord tc{b0 * uv[0].x + b1 * uv[1].x + b2 * uv[2].x, b0 * uv[0].y + b1 * uv[1].y + b2 * uv[2].y, 0.f, 0.f, 0.f, 0.f};
    if (tex_f32(sc, (int)(meta2 >> 9), tc) == 0.0f) return true;
  }
  return false;
}
// inline fast path: no alpha mask and a triangle of non-zero area can never be rejected here
PT_DEV bool tri_post_reject(const DevScene& sc, int prim, V3 p0, V3 p1, V3 p2, uint32_t meta2, float b0, float b1, float b2, bool closest) {
  const bool has_alpha = (meta2 & PT_TRI_ALPHA_BIT) != 0;
  if (!closest && !has_alpha) return false;
  if (!has_alpha) {
    V3 ng = cross(p2 - p0, p1 - p0);
    if (norm_squared(ng) != 0.0f) return false;
  }
  return tri_post_reject_slow(sc, prim, p0, p1, p2, meta2, b0, b1, b2);
}

struct NodeLoad {
  float4 a, b;  // a = (min.x, min.y, min.z, max.x)  b = (max.y, max.z, offset bits, n_prims | axis << 16)
};
// One 32 B node as a single 256-bit non-coherent load (LDG.E.256 on sm_100a).
PT_DEV NodeLoad load_node(const float4* __restrict__ nodes, uint32_t i) {
  NodeLoad n;
  asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(n.a.x), "=f"(n.a.y), "=f"(n.a.z), "=f"(n.a.w), "=f"(n.b.x), "=f"(n.b.y), "=f"(n.b.z), "=f"(n.b.w)
      : "l"(nodes + 2 * (size_t)i));
  return n;
}

// 3-input min / max (FMNMX3 on sm_100a).  A NaN operand is ignored, as in the 2-input forms.
PT_DEV float fmax3_nn(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
PT_DEV float fmin3_nn(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// Two node records in ONE asm statement: both loads are issued before anything waits on the first (left to itself the
// register allocator may give the second load the registers the first record's slab test is still reading, which
// serialises two DRAM round trips per traversal step: measured +17 % on the 10 M-triangle tree with incoherent rays).
#ifndef PT_PAIR_LOAD128
#define PT_PAIR_LOAD128 1
#endif
#ifndef PT_NODE_EVICT_LAST
#define PT_NODE_EVICT_LAST 0
#endif
PT_DEV void load_node_pair(const float4* __restrict__ nodes, uint32_t ia, uint32_t ib, NodeLoad* a, NodeLoad* b) {
#if PT_PAIR_LOAD128
  // four 128-bit loads, the first half of either record first: with 64 registers per thread the allocator keeps three of
  // them in flight and re-uses the first one's registers for the fourth — which by then is an L1 hit, because the two
  // halves of a 32-byte record are one sector.  Two 256-bit loads get serialised instead (the second one is given the
  // registers the first record's slab test is still reading): two DRAM round trips per step on trees beyond L2 size.
  const float4* pa = nodes + 2 * (size_t)ia;
  const float4* pb = nodes + 2 * (size_t)ib;
#if PT_NODE_EVICT_LAST
  // node lines are asked to stay: the second half of a record may be read a few dozen instructions after the first
  auto ld = [](const float4* p) {
    float4 v;
    asm("ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
  };
  a->a = ld(pa);
  b->a = ld(pb);
  a->b = ld(pa + 1);
  b->b = ld(pb + 1);
#else
  a->a = __ldg(pa);
  b->a = __ldg(pb);
  a->b = __ldg(pa + 1);
  b->b = __ldg(pb + 1);
#endif
#else
  *a = load_node(nodes, ia);
  *b = load_node(nodes, ib);
#endif
}

// bounds.rs:190-232.  The slab arithmetic does not depend on the ray's current t_max except for the
// final `t_min < r.t_max`, so it is split: box_geom() returns the geometric part and the entry distance,
// and the caller applies `t_entry < t_max` with whatever t_max is current when the reference would have
// run the test.
//
// The six plane distances are the reference's expressions, operation for operation.  Its compare-and-select
// chains over them are folded into one 3-input max and one 3-input min, which decides the same for every input
// (tests/test_slab_formulations.py sweeps 10^7 adversarial cases incl. NaN, infinities, signed zeros):
//  * the reference misses iff some near-plane distance exceeds another axis' (widened) far-plane distance; the
//    same-axis pairs the max / min form also compares can only fire when that far distance is negative, where
//    `t_max > 0` rejects anyway;
//  * x -> fl(x * g) is monotonic, so widening after the min equals the min of the widened values, bit for bit;
//  * a NaN (0 * inf: origin on a slab plane of an axis the ray is parallel to) never compares true, so in the
//    reference's chains one that enters the accumulators from the x axis sticks and rejects at `t_min < r.t_max` /
//    `t_max > 0`, one from y or z is passed over; min / max pass over every NaN, hence the explicit test on x.
// t_entry equals the reference's t_min wherever the box is accepted (up to the sign of a zero).
PT_DEV bool box_geom(const NodeLoad& n, V3 o, V3 inv_dir, bool nx, bool ny, bool nz, float* t_entry) {
  const float g = 1.0f + 2.0f * gamma_n(3);
  const float tx_min = ((nx ? n.a.w : n.a.x) - o.x) * inv_dir.x;
  const float tx_max = ((nx ? n.a.x : n.a.w) - o.x) * inv_dir.x;
  const float ty_min = ((ny ? n.b.x : n.a.y) - o.y) * inv_dir.y;
  const float ty_max = ((ny ? n.a.y : n.b.x) - o.y) * inv_dir.y;
  const float tz_min = ((nz ? n.b.y : n.a.z) - o.z) * inv_dir.z;
  const float tz_max = ((nz ? n.a.z : n.b.y) - o.z) * inv_dir.z;
  const float t_min = fmax3_nn(tx_min, ty_min, tz_min);
  const float t_max = fmin3_nn(tx_max, ty_max, tz_max) * g;
  *t_entry = t_min;
  return !(t_min > t_max) & (t_max > 0.0f) & (tx_min == tx_min) & (tx_max == tx_max);
}

// The slab tests of both children of a node, written plane by plane over the two records so that every record is needed
// from the first operation on: both loads have to be in flight before anything is computed.
PT_DEV void box_geom_pair(const NodeLoad& a, const NodeLoad& b, V3 o, V3 inv_dir, bool nx, bool ny, bool nz, bool* ga, float* ta, bool* gb,
                          float* tb) {
  const float g = 1.0f + 2.0f * gamma_n(3);
  const float ax0 = ((nx ? a.a.w : a.a.x) - o.x) * inv_dir.x, bx0 = ((nx ? b.a.w : b.a.x) - o.x) * inv_dir.x;
  const float ax1 = ((nx ? a.a.x : a.a.w) - o.x) * inv_dir.x, bx1 = ((nx ? b.a.x : b.a.w) - o.x) * inv_dir.x;
  const float ay0 = ((ny ? a.b.x : a.a.y) - o.y) * inv_dir.y, by0 = ((ny ? b.b.x : b.a.y) - o.y) * inv_dir.y;
  const float ay1 = ((ny ? a.a.y : a.b.x) - o.y) * inv_dir.y, by1 = ((ny ? b.a.y : b.b.x) - o.y) * inv_dir.y;
  const float az0 = ((nz ? a.b.y : a.a.z) - o.z) * inv_dir.z, bz0 = ((nz ? b.b.y : b.a.z) - o.z) * inv_dir.z;
  const float az1 = ((nz ? a.a.z : a.b.y) - o.z) * inv_dir.z, bz1 = ((nz ? b.a.z : b.b.y) - o.z) * inv_dir.z;
  const float a_min = fmax3_nn(ax0, ay0, az0), b_min = fmax3_nn(bx0, by0, bz0);
  const float a_max = fmin3_nn(ax1, ay1, az1) * g, b_max = fmin3_nn(bx1, by1, bz1) * g;
  *ta = a_min;
  *tb = b_min;
  *ga = !(a_min > a_max) & (a_max > 0.0f) & (ax0 == ax0) & (ax1 == ax1);
  *gb = !(b_min > b_max) & (b_max > 0.0f) & (bx0 == bx0) & (bx1 == bx1);
}

#define PT_STACK_SIZE 64
// "no node in hand".  A node's meta word is n_prims | axis << 16 (bits 18..31 clear), so with this value one masked test
// tells the three cases apart: leaf = low 16 bits non-zero, interior = (meta & 0x8000ffff) == 0, none = bit 31.
#define PT_NO_NODE 0x80000000u
#define PT_IS_LEAF(m) (((m) & 0xffffu) != 0u)
#define PT_IS_INTERIOR(m) (((m) & 0x8000ffffu) == 0u)

// ------------------------------------------------------------------------------------------------------
// Device node order.  ptrs_scene_create() keeps the reference's 32-byte LinearBVHNode records but stores
// the two children of every interior node SIDE BY SIDE (one 64-byte, 64-byte-aligned pair; the root sits
// alone in slot 0, slot 1 is padding), pairs in depth-first order.  An interior node's `offset` is the
// index of its first (left) child, the second child is offset + 1.  One traversal step therefore fetches
// one contiguous 64 B block instead of two unrelated 32 B records.  Boxes, split axes, leaf ranges and
// therefore the visit order are exactly those of accelerator.rs:348-357's flattened tree.
//
// Streaming traversal engine for the bulk kernels.
//
// A warp owns 32 ray slots.  Each lane takes ITS ray through the box-test / triangle-test decisions of
// accelerator.rs:359-475, with:
//   refill     lanes whose ray has ended pull new work items with ONE atomicAdd for the whole warp
//              (persistent threads, warp-aggregated fetch) as soon as PT_REFILL_IDLE lanes are idle
//   expand     a lane standing on an interior node loads BOTH children and runs both slab tests.  The
//              near child (dir_is_neg[axis]) is accepted against t_max; the far child's entry distance goes
//              on the stack, and `t_entry < t_max` is applied again when it is popped — the very test the
//              reference performs at that moment, since only that comparison depends on t_max
//   postpone   (fast variant) a lane that reaches a leaf parks it and keeps descending until it holds a
//              second leaf; the warp switches to the triangle phase when fewer than box_min (DevScene, 12 or 20) lanes can
//              still take a box step.  Exactness: with nested boxes the slab entry distance can only grow
//              from a node to its descendants (float subtraction and multiplication are monotonic), so a
//              node accepted under a stale (larger) t_max that the reference would have culled can only
//              lead to leaves whose own entry distance fails the CURRENT t_max — and every parked node is
//              re-validated with `t_entry < t_max` whenever a hit shrinks t_max, every stack entry when
//              it is popped.  Leaves are processed first-in first-out, so each triangle is tested in the
//              reference's order against the reference's t_max: hits, ties and barycentrics are identical.
// Stack entries are 16 B {entry distance, offset, n_prims | axis << 16, -}: a pop needs no node reload.
//
// Work is a functor object with
//   bool begin(uint32_t item, LaneRay* r)                       first ray of a work item (false: nothing to trace)
//   bool end(uint32_t item, const DevHit& h, bool found, LaneRay* r)   ray ended; true = trace *r next for the same item
// ------------------------------------------------------------------------------------------------------
struct LaneRay {
  V3 o, d;
  float t_max;
  bool any_hit;
};

#ifndef PT_REFILL_IDLE
#define PT_REFILL_IDLE 8
#endif
#ifndef PT_SEARCH_MIN
#define PT_SEARCH_MIN 6
#endif

// empty accelerator: every ray misses (accelerator.rs:360-362)
template <class Work>
PT_DEV void trace_empty(uint32_t n_items, uint32_t* ticket, Work& work) {
  DevHit miss;
  miss.prim = -1;
  miss.t = miss.b0 = miss.b1 = miss.b2 = 0.f;
  const int lane = threadIdx.x & 31;
  for (;;) {
    const uint32_t base = (lane == 0) ? atomicAdd(ticket, 32u) : 0u;
    const uint32_t b = __shfl_sync(0xffffffffu, base, 0);
    if (b >= n_items) return;
    const uint32_t i = b + lane;
    if (i < n_items) {
      LaneRay r;
      bool more = work.begin(i, &r);
      while (more) more = work.end(i, miss, false, &r);
    }
  }
}

// ---- fast variant (no visit counters): box loop, then triangle loop, then service -------------------------
// Register diet (the kernels run at 64 registers / 32 warps per SM): the per-ray booleans and the triangle
// test's axis live in ONE word, the hit distance is t_max itself, "found" is hit_prim >= 0, and the parked
// leaf is (next primitive, triangles left).
#define PT_RB_NX 1u
#define PT_RB_NY 2u
#define PT_RB_NZ 4u
#define PT_RB_KZ_SHIFT 3
#define PT_RB_ANY 32u
#define PT_RB_LIVE 64u
// box steps per scheduling decision (measured on B200, round 2: 1 -> 3 steps takes 3 % off the traversal kernels on every
// scene; 4 is level with 3)
#ifndef PT_BOX_STEPS
#define PT_BOX_STEPS 3
#endif
#ifndef PT_TRI_STEPS
#define PT_TRI_STEPS 1
#endif
// PT_EAGER_POP: a lane that is left without a node pops its next stack entry at the END of the step (one predicated
// 16-byte local load in the convergent instruction stream) and the entry's `t_entry < t_max` test — the reference's box
// test at pop time — is made when the node is used, together with the re-validation every node in hand needs anyway after
// a hit has shrunk t_max.  Replaces the divergent pop section at the top of the step.
#ifndef PT_EAGER_POP
#define PT_EAGER_POP 0
#endif
#ifndef PT_NEAR_LEAF_DIRECT
#define PT_NEAR_LEAF_DIRECT 0
#endif
// PT_SMEM_STACK = K: the K entries nearest the bottom of every ray's pending stack live in shared memory, one 16-byte
// column per thread ([level][thread], so a warp's access is conflict-free whatever levels its lanes stand on: four
// wavefronts, where the same access to thread-interleaved local memory touches four 128-byte lines PER DISTINCT LEVEL
// among the lanes); deeper entries stay in local memory.  Blocks of PT_TRACE_BLOCK threads.
#ifndef PT_SMEM_STACK
#define PT_SMEM_STACK 0
#endif
#ifndef PT_STACK8
#define PT_STACK8 0
#endif
#ifndef PT_PUSH_PREFETCH
#define PT_PUSH_PREFETCH 0
#endif
// PT_PARK_PREFETCH_ON: when a leaf is parked its first triangle is requested into L1 — unlike a pushed node a parked leaf is
// always processed, and until then the lane keeps taking box steps
#ifndef PT_PARK_PREFETCH_ON
#define PT_PARK_PREFETCH_ON 0
#endif
#if PT_PARK_PREFETCH_ON
#define PT_PARK_PREFETCH(prim) asm volatile("prefetch.global.L1 [%0];" ::"l"(sc.tri_verts + 3 * (size_t)(prim)))
#else
#define PT_PARK_PREFETCH(prim) ((void)0)
#endif

#ifndef PT_TRACE_BLOCK
#define PT_TRACE_BLOCK 128
#endif
// DIST: of two entered children the one the ray enters first is visited first (trees the library built itself) instead of
// dir_is_neg[axis] (the reference's order on the reference's tree).  A template parameter, so that the reference path's
// code is untouched.
template <bool DIST, class Work>
PT_DEV void trace_fast(const DevScene& sc, uint32_t n_items, uint32_t* ticket, Work& work) {
  if (sc.n_nodes == 0) {
    trace_empty(n_items, ticket, work);
    return;
  }
  const uint32_t FULL = 0xffffffffu;
  // fewer lanes than this able to take a box step -> the warp turns to its parked leaves.  Scheduling only (results do
  // not depend on it); measured: 12 is best on trees of a few dozen nodes, 20 on trees of 10^5 .. 10^7 nodes.
  const int box_min = (int)sc.box_min;
  const bool pop_twice = sc.pop_twice != 0;
  constexpr bool dist_order = DIST;
#if PT_STACK8
  // 8-byte entries {entry distance, packed node}: half the local-memory footprint of the 1024 stacks per SM, which is what
  // matters when the tree itself does not fit in L2 and the stacks compete with its nodes for L1.  Packed node word:
  //   bit 31 = 0              interior: first child slot (even, < 2^30) << 1 | split axis
  //   bit 31 = 1, bit 30 = 0  leaf: (n_prims - 1) << 26 | first primitive      (n_prims <= 16, primitive < 2^26)
  //   bit 31 = 1, bit 30 = 1  leaf by reference: the node's slot; (offset, n_prims) are re-read when it is popped
  uint2 stack[PT_STACK_SIZE];
  auto st_load = [&](int i, float* t, uint32_t* off, uint32_t* meta) {
    const uint2 e = stack[i];
    *t = __uint_as_float(e.x);
    const uint32_t w = e.y;
    if (!(w & 0x80000000u)) {
      *off = (w & ~3u) >> 1;
      *meta = (w & 3u) << 16;
    } else if (!(w & 0x40000000u)) {
      *off = w & 0x03ffffffu;
      *meta = ((w >> 26) & 15u) + 1u;
    } else {
      const float2 om = __ldg(reinterpret_cast<const float2*>(sc.nodes + 2 * (size_t)(w & 0x3fffffffu) + 1) + 1);
      *off = __float_as_uint(om.x);
      *meta = __float_as_uint(om.y);
    }
  };
  auto st_store = [&](int i, float t, uint32_t off, uint32_t meta, uint32_t slot) {
    const uint32_t np = meta & 0xffffu;
    uint32_t w;
    if (np == 0u) w = (off << 1) | ((meta >> 16) & 3u);
    else if (np <= 16u && off < (1u << 26)) w = 0x80000000u | ((np - 1u) << 26) | off;
    else w = 0xc0000000u | slot;
    stack[i] = make_uint2(__float_as_uint(t), w);
  };
#elif PT_SMEM_STACK
  __shared__ uint4 sm_stack[PT_SMEM_STACK * PT_TRACE_BLOCK];
  uint4 stack[PT_STACK_SIZE - PT_SMEM_STACK];
  auto st_load = [&](int i, float* t, uint32_t* off, uint32_t* meta) {
    const uint4 e = i < PT_SMEM_STACK ? sm_stack[i * PT_TRACE_BLOCK + threadIdx.x] : stack[i - PT_SMEM_STACK];
    *t = __uint_as_float(e.x);
    *off = e.y;
    *meta = e.z;
  };
  auto st_store = [&](int i, float t, uint32_t off, uint32_t meta, uint32_t) {
    const uint4 e = make_uint4(__float_as_uint(t), off, meta, 0u);
    if (i < PT_SMEM_STACK) sm_stack[i * PT_TRACE_BLOCK + threadIdx.x] = e;
    else stack[i - PT_SMEM_STACK] = e;
  };
#else
  uint4 stack[PT_STACK_SIZE];
  auto st_load = [&](int i, float* t, uint32_t* off, uint32_t* meta) {
    const uint4 e = stack[i];
    *t = __uint_as_float(e.x);
    *off = e.y;
    *meta = e.z;
  };
  auto st_store = [&](int i, float t, uint32_t off, uint32_t meta, uint32_t) { stack[i] = make_uint4(__float_as_uint(t), off, meta, 0u); };
#endif
  int sp_ = 0;
  // node in hand (its box test passed under the t_max current at that time): offset, meta, entry distance
  uint32_t cur_off = 0, cur_meta = PT_NO_NODE;
  float cur_t = 0.f;
  uint32_t pl_off = 0, pl_cnt = 0;  // parked leaf: next primitive, triangles left (0 = none)
  uint32_t rbits = 0;               // PT_RB_*
  bool exhausted = n_items == 0;
  uint32_t item = 0;
  V3 o = mk3(0, 0, 0), inv_dir = mk3(0, 0, 0);
  float sx = 0.f, sy = 0.f, sz = 0.f;
  float t_max = 0.f;
  int hit_prim = -1;
  float hit_b0 = 0.f, hit_b1 = 0.f, hit_b2 = 0.f;

  auto start_ray = [&](const LaneRay& r) {
    o = r.o;
    inv_dir = mk3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z);
    const RayPre rp = ray_precompute(r.d);
    sx = rp.sx;
    sy = rp.sy;
    sz = rp.sz;
    rbits = PT_RB_LIVE | (inv_dir.x < 0.0f ? PT_RB_NX : 0u) | (inv_dir.y < 0.0f ? PT_RB_NY : 0u) | (inv_dir.z < 0.0f ? PT_RB_NZ : 0u) |
            ((uint32_t)rp.kz << PT_RB_KZ_SHIFT) | (r.any_hit ? PT_RB_ANY : 0u);
    t_max = r.t_max;
    hit_prim = -1;
    hit_b0 = hit_b1 = hit_b2 = 0.f;
    sp_ = 0;
    pl_cnt = 0;
    // root: tested like any other node (accelerator.rs:372-374)
    const NodeLoad n = load_node(sc.nodes, 0);
    float te;
    if (box_geom(n, o, inv_dir, rbits & PT_RB_NX, rbits & PT_RB_NY, rbits & PT_RB_NZ, &te) && te < t_max) {
      cur_off = __float_as_uint(n.b.z);
      cur_meta = __float_as_uint(n.b.w);
      cur_t = te;
    } else {
      cur_meta = PT_NO_NODE;
    }
  };

  for (;;) {
    // ---- refill ------------------------------------------------------------------------------------
    const uint32_t idle = __ballot_sync(FULL, !(rbits & PT_RB_LIVE));
    if (!exhausted && (__popc(idle) >= PT_REFILL_IDLE)) {
      const int lane = threadIdx.x & 31;
      const int leader = __ffs(idle) - 1;
      uint32_t base = 0;
      if (lane == leader) base = atomicAdd(ticket, (uint32_t)__popc(idle));
      base = __shfl_sync(FULL, base, leader);
      if (base + (uint32_t)__popc(idle) >= n_items) exhausted = true;
      if (!(rbits & PT_RB_LIVE)) {
        const uint32_t i = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
        if (i < n_items) {
          LaneRay r;
          if (work.begin(i, &r)) {
            item = i;
            start_ray(r);
          }
        }
      }
    }
    if (__ballot_sync(FULL, rbits & PT_RB_LIVE) == 0) {
      if (exhausted) break;
      continue;
    }

    // ---- box phase: pop / park / expand ----------------------------------------------------------------
#if PT_EAGER_POP
    auto eager_pop = [&]() {
      if ((rbits & PT_RB_LIVE) && cur_meta == PT_NO_NODE && sp_ > 0) {
        --sp_;
        st_load(sp_, &cur_t, &cur_off, &cur_meta);
      }
    };
    auto box_step = [&]() {
      const bool live = (rbits & PT_RB_LIVE) != 0;
      // the node in hand under the current t_max: the reference's box test at pop time, and the re-test a node accepted
      // before a hit needs
      if (cur_meta != PT_NO_NODE && !(cur_t < t_max)) cur_meta = PT_NO_NODE;
#if PT_EAGER_POP == 2
      // the entry popped ahead was culled: one more pop, tested on the spot, so that the lane still expands a node in this step
      if (live && cur_meta == PT_NO_NODE && sp_ > 0) {
        --sp_;
        float et;
        uint32_t eo, em;
        st_load(sp_, &et, &eo, &em);
        if (et < t_max) {
          cur_t = et;
          cur_off = eo;
          cur_meta = em;
        }
      }
#endif
      if (live && cur_meta != PT_NO_NODE) {
        if ((cur_meta & 0xffffu) != 0) {
          if (pl_cnt == 0) {  // park the leaf, keep descending
            pl_off = cur_off;
            pl_cnt = cur_meta & 0xffffu;
            cur_meta = PT_NO_NODE;
          }
        } else {
          const NodeLoad L = load_node(sc.nodes, cur_off);
          const NodeLoad R = load_node(sc.nodes, cur_off + 1);
          const bool nx = rbits & PT_RB_NX, ny = rbits & PT_RB_NY, nz = rbits & PT_RB_NZ;
          float tl, tr;
          const bool gl = box_geom(L, o, inv_dir, nx, ny, nz, &tl);
          const bool gr = box_geom(R, o, inv_dir, nx, ny, nz, &tr);
          const bool neg = dist_order ? (tr < tl) : (((rbits >> ((cur_meta >> 16) & 3u)) & 1u) != 0);  // dir_is_neg[axis], or nearer child first
          // near child first (accelerator.rs:393-404)
          const bool gn = neg ? gr : gl, gf = neg ? gl : gr;
          const float tn = neg ? tr : tl, tf = neg ? tl : tr;
          const float4 nb = neg ? R.b : L.b, fb = neg ? L.b : R.b;
          bool an = gn && tn < t_max;
          const bool af = gf && tf < t_max;
          // an entered near child that is a leaf goes straight to the free parking slot; the far child is then the node
          // in hand without a push / pop pair
          if (an && (__float_as_uint(nb.w) & 0xffffu) != 0u && pl_cnt == 0u) {
            pl_off = __float_as_uint(nb.z);
            pl_cnt = __float_as_uint(nb.w) & 0xffffu;
            an = false;
          }
          if (af && !an) {
            cur_t = tf;
            cur_off = __float_as_uint(fb.z);
            cur_meta = __float_as_uint(fb.w);
          } else {
            if (af) {
              if (sp_ < PT_STACK_SIZE) {  // always true: ptrs_scene_create refuses trees deeper than the stack
                st_store(sp_, tf, __float_as_uint(fb.z), __float_as_uint(fb.w), cur_off + (neg ? 0u : 1u));
                ++sp_;
              }
            }
            if (an) {
              cur_t = tn;
              cur_off = __float_as_uint(nb.z);
              cur_meta = __float_as_uint(nb.w);
            } else {
              cur_meta = PT_NO_NODE;
            }
          }
          // the node now in hand is a leaf and the parking slot is free: park it here instead of in the next iteration
          if (cur_meta != PT_NO_NODE && (cur_meta & 0xffffu) != 0u && pl_cnt == 0u) {
            pl_off = cur_off;
            pl_cnt = cur_meta & 0xffffu;
            cur_meta = PT_NO_NODE;
          }
        }
      }
      eager_pop();
    };
#else
    // (a lane without a ray has no node in hand, an empty stack and no parked leaf, so none of the tests below asks for
    // PT_RB_LIVE on top)
    auto box_step = [&]() {
      const bool cur_leaf = PT_IS_LEAF(cur_meta);
      const bool can_box = PT_IS_INTERIOR(cur_meta) || (cur_meta == PT_NO_NODE && sp_ > 0) || (cur_leaf && pl_cnt == 0);
      if (can_box) {
        if (cur_meta == PT_NO_NODE) {  // pop one entry; the reference's box test at pop time
          --sp_;
          float et;
          uint32_t eo, em;
          st_load(sp_, &et, &eo, &em);
          if (et < t_max) {
            cur_t = et;
            cur_off = eo;
            cur_meta = em;
          }
          if (pop_twice) {
            // the entry was culled, or it was a leaf that goes straight to the free parking slot: one more pop (at most),
            // so that the lane still has a node to expand in this iteration.  Pays on trees that do not fit in L1
            // (scheduling only; DevScene::pop_twice)
            if (PT_IS_LEAF(cur_meta) && pl_cnt == 0u) {
              pl_off = cur_off;
              PT_PARK_PREFETCH(cur_off);
              pl_cnt = cur_meta & 0xffffu;
              cur_meta = PT_NO_NODE;
            }
            if (cur_meta == PT_NO_NODE && sp_ > 0) {
              --sp_;
              st_load(sp_, &et, &eo, &em);
              if (et < t_max) {
                cur_t = et;
                cur_off = eo;
                cur_meta = em;
              }
            }
          }
        }
        if (cur_meta != PT_NO_NODE) {
          if ((cur_meta & 0xffffu) != 0) {
            if (pl_cnt == 0) {  // park the leaf, keep descending
              pl_off = cur_off;
              PT_PARK_PREFETCH(cur_off);
              pl_cnt = cur_meta & 0xffffu;
              cur_meta = PT_NO_NODE;
            }
          } else {
            // dir_is_neg straight from the sign of inv_dir (what PT_RB_N* were set from): compares on registers that are live
            // anyway instead of three more registers holding the extracted bits
            const bool nx = inv_dir.x < 0.0f, ny = inv_dir.y < 0.0f, nz = inv_dir.z < 0.0f;
            // which child first: dir_is_neg[axis] on a reference-built tree (the reference's order, accelerator.rs:393-404) —
            // known before the fetch, so the two records are loaded as (near, far) and nothing is swapped afterwards; on a
            // tree the library built itself the child the ray enters first
            bool neg = ((rbits >> (cur_meta >> 16)) & 1u) != 0;  // (an interior node's meta word is axis << 16, nothing else)
            const uint32_t first = dist_order ? 0u : (neg ? 1u : 0u);
            NodeLoad A, B;
            load_node_pair(sc.nodes, cur_off + first, cur_off + (first ^ 1u), &A, &B);
            float ta, tb;
            bool ga, gb;
            box_geom_pair(A, B, o, inv_dir, nx, ny, nz, &ga, &ta, &gb, &tb);
            if (dist_order) neg = tb < ta;
            const bool swap = dist_order && neg;
            const bool gn = swap ? gb : ga, gf = swap ? ga : gb;
            const float tn = swap ? tb : ta, tf = swap ? ta : tb;
            const float4 nb = swap ? B.b : A.b, fb = swap ? A.b : B.b;
            bool an = gn && tn < t_max;
            const bool af = gf && tf < t_max;
#if PT_NEAR_LEAF_DIRECT
            // an entered near child that is a leaf goes straight to the free parking slot; the far child is then the node in
            // hand without a push / pop pair
            if (an && (__float_as_uint(nb.w) & 0xffffu) != 0u && pl_cnt == 0u) {
              pl_off = __float_as_uint(nb.z);
              pl_cnt = __float_as_uint(nb.w) & 0xffffu;
              an = false;
            }
#endif
            if (af && !an) {
              // near child rejected, far child entered: the reference pushes the far child and pops it straight away; the
              // pop's re-test against t_max is what the node in hand gets anyway whenever a hit shrinks t_max
              cur_t = tf;
              cur_off = __float_as_uint(fb.z);
              cur_meta = __float_as_uint(fb.w);
            } else {
              if (af) {
                if (sp_ < PT_STACK_SIZE) {  // always true: ptrs_scene_create refuses trees deeper than the stack
                  st_store(sp_, tf, __float_as_uint(fb.z), __float_as_uint(fb.w), cur_off + (neg ? 0u : 1u));
                  ++sp_;
#if PT_PUSH_PREFETCH
                  // the pushed child's own children (or its first triangle): requested now, so that the pop finds them in
                  // L1 / L2 instead of starting the round trip then
                  {
                    const uint32_t fo = __float_as_uint(fb.z);
                    const void* pf = (__float_as_uint(fb.w) & 0xffffu) ? (const void*)(sc.tri_verts + 3 * (size_t)fo) : (const void*)(sc.nodes + 2 * (size_t)fo);
#if PT_PUSH_PREFETCH == 2
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
#else
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(pf));
#endif
                  }
#endif
                }
              }
              if (an) {
                cur_t = tn;
                cur_off = __float_as_uint(nb.z);
                cur_meta = __float_as_uint(nb.w);
              } else {
                cur_meta = PT_NO_NODE;
              }
            }
            // the node now in hand is a leaf and the parking slot is free: park it here instead of in the next iteration
            if (PT_IS_LEAF(cur_meta) && pl_cnt == 0u) {
              pl_off = cur_off;
              PT_PARK_PREFETCH(cur_off);
              pl_cnt = cur_meta & 0xffffu;
              cur_meta = PT_NO_NODE;
            }
          }
        }
      }
    };
#endif
    for (;;) {
      const bool live = (rbits & PT_RB_LIVE) != 0;
      const bool cur_leaf = PT_IS_LEAF(cur_meta);
#if PT_EAGER_POP
      const bool can_box = live && cur_meta != PT_NO_NODE && (!cur_leaf || pl_cnt == 0);  // no node in hand => empty stack
#else
      const bool can_box = PT_IS_INTERIOR(cur_meta) || (cur_meta == PT_NO_NODE && sp_ > 0) || (cur_leaf && pl_cnt == 0);
#endif
      const uint32_t bmask = __ballot_sync(FULL, can_box);
      if (bmask == 0) break;
      if (__popc(bmask) < box_min && __ballot_sync(FULL, live && !can_box) != 0) break;
      // PT_BOX_STEPS steps under one scheduling decision: the ballots and the phase test are paid once per group of steps
#pragma unroll
      for (int rep = 0; rep < PT_BOX_STEPS; ++rep) box_step();
    }

    // ---- triangle phase: parked leaves, first in first out -----------------------------------------------
    auto tri_step = [&]() {
#if PT_EAGER_POP
      const bool live = (rbits & PT_RB_LIVE) != 0;
      if (live && pl_cnt == 0 && cur_meta != PT_NO_NODE && (cur_meta & 0xffffu) != 0) {  // second leaf moves up, if it still qualifies
        if (cur_t < t_max) {
          pl_off = cur_off;
          pl_cnt = cur_meta & 0xffffu;
        }
        cur_meta = PT_NO_NODE;
      }
#else
      if (pl_cnt == 0 && PT_IS_LEAF(cur_meta)) {  // second leaf moves up
        pl_off = cur_off;
        pl_cnt = cur_meta & 0xffffu;
        cur_meta = PT_NO_NODE;
      }
#endif
      if (pl_cnt != 0) {
        const uint32_t prim = pl_off;
        const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim);
        const float4 v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1);
        const float4 v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
        ++pl_off;
        --pl_cnt;
        RayPre rp;
        rp.kz = (int)((rbits >> PT_RB_KZ_SHIFT) & 3u);
        rp.sx = sx;
        rp.sy = sy;
        rp.sz = sz;
        float t, b0, b1, b2;
        if (tri_core(mk3(v0), mk3(v1), mk3(v2), o, rp, t_max, &t, &b0, &b1, &b2) &&
            !tri_post_reject(sc, (int)prim, mk3(v0), mk3(v1), mk3(v2), __float_as_uint(v2.w), b0, b1, b2, !(rbits & PT_RB_ANY))) {
          hit_prim = (int)prim;
          hit_b0 = b0;
          hit_b1 = b1;
          hit_b2 = b2;
          t_max = t;
          if (rbits & PT_RB_ANY) {  // intersect_p returns at the first hit (accelerator.rs:435-442)
            pl_cnt = 0;
            sp_ = 0;
            cur_meta = PT_NO_NODE;
          }
#if !PT_EAGER_POP
          else if (cur_meta != PT_NO_NODE && !(cur_t < t_max)) {
            cur_meta = PT_NO_NODE;  // the node in hand was accepted under the old t_max: re-validate
          }
#endif
        }
      }
#if PT_EAGER_POP
      eager_pop();
#endif
    };
    for (;;) {
      const bool has = pl_cnt != 0 || PT_IS_LEAF(cur_meta);
      if (__ballot_sync(FULL, has) == 0) break;
#pragma unroll
      for (int rep = 0; rep < PT_TRI_STEPS; ++rep) tri_step();
    }

    // ---- rays that ran out of nodes --------------------------------------------------------------------
    if ((rbits & PT_RB_LIVE) && cur_meta == PT_NO_NODE && sp_ == 0 && pl_cnt == 0) {
      DevHit h;
      h.prim = hit_prim;
      h.t = t_max;
      h.b0 = hit_b0;
      h.b1 = hit_b1;
      h.b2 = hit_b2;
      LaneRay r;
      if (work.end(item, h, hit_prim >= 0, &r)) start_ray(r);
      else rbits = 0;
    }
  }
}

// ---- counting variant: strictly the reference's node-test sequence (no postponed leaves), so that the
// node / triangle test counters equal the CPU path's ------------------------------------------------------
template <class Work>
PT_DEV void trace_counted(const DevScene& sc, uint32_t n_items, uint32_t* ticket, Work& work, uint32_t* c_nodes, uint32_t* c_tris) {
  if (sc.n_nodes == 0) {
    trace_empty(n_items, ticket, work);
    return;
  }
  const uint32_t FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const uint32_t lane_lt = (1u << lane) - 1u;
  uint4 stack[PT_STACK_SIZE];
  int sp_ = 0;
  uint32_t cur_off = 0, cur_meta = PT_NO_NODE;
  bool active = false, exhausted = n_items == 0, done_ray = false;
  bool any_hit = false, found = false;
  uint32_t item = 0;
  V3 o = mk3(0, 0, 0), inv_dir = mk3(0, 0, 0);
  bool nx = false, ny = false, nz = false;
  RayPre rp = ray_precompute(mk3(0, 0, 1));
  float t_max = 0.f;
  DevHit hit;
  hit.prim = -1;
  hit.t = hit.b0 = hit.b1 = hit.b2 = 0.f;

  auto start_ray = [&](const LaneRay& r) {
    o = r.o;
    inv_dir = mk3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z);
    nx = inv_dir.x < 0.0f;
    ny = inv_dir.y < 0.0f;
    nz = inv_dir.z < 0.0f;
    rp = ray_precompute(r.d);
    t_max = r.t_max;
    any_hit = r.any_hit;
    found = false;
    hit.prim = -1;
    hit.t = r.t_max;
    hit.b0 = hit.b1 = hit.b2 = 0.f;
    sp_ = 0;
    done_ray = false;
    const NodeLoad n = load_node(sc.nodes, 0);
    ++*c_nodes;
    float te;
    if (box_geom(n, o, inv_dir, nx, ny, nz, &te) && te < t_max) {
      cur_off = __float_as_uint(n.b.z);
      cur_meta = __float_as_uint(n.b.w);
    } else {
      cur_meta = PT_NO_NODE;
      done_ray = true;
    }
  };

  for (;;) {
    const uint32_t idle = __ballot_sync(FULL, !active);
    if (!exhausted && (__popc(idle) >= PT_REFILL_IDLE)) {
      const int leader = __ffs(idle) - 1;
      uint32_t base = 0;
      if (lane == leader) base = atomicAdd(ticket, (uint32_t)__popc(idle));
      base = __shfl_sync(FULL, base, leader);
      if (base + (uint32_t)__popc(idle) >= n_items) exhausted = true;
      if (!active) {
        const uint32_t i = base + (uint32_t)__popc(idle & lane_lt);
        if (i < n_items) {
          LaneRay r;
          if (work.begin(i, &r)) {
            item = i;
            active = true;
            start_ray(r);
          }
        }
      }
    }
    if (__ballot_sync(FULL, active) == 0) {
      if (exhausted) break;
      continue;
    }
    // phase A: descend until a leaf is in hand
    for (;;) {
      if (active && !done_ray && cur_meta == PT_NO_NODE) {
        for (;;) {  // pop until an entry survives the t_max test (the reference's box test at pop time)
          if (sp_ == 0) {
            done_ray = true;
            break;
          }
          --sp_;
          const uint4 e = stack[sp_ < PT_STACK_SIZE ? sp_ : PT_STACK_SIZE - 1];
          ++*c_nodes;
          if (__uint_as_float(e.x) < t_max) {
            cur_off = e.y;
            cur_meta = e.z;
            break;
          }
        }
      }
      const bool is_leaf = (cur_meta & 0xffffu) != 0;
      const bool search = active && !done_ray && cur_meta != PT_NO_NODE && !is_leaf;
      const uint32_t smask = __ballot_sync(FULL, search);
      if (smask == 0) break;
      const uint32_t lmask = __ballot_sync(FULL, active && !done_ray && cur_meta != PT_NO_NODE && is_leaf);
      if (lmask != 0 && __popc(smask) < PT_SEARCH_MIN) break;
      if (search) {
        const NodeLoad L = load_node(sc.nodes, cur_off);
        const NodeLoad R = load_node(sc.nodes, cur_off + 1);
        const uint32_t axis = (cur_meta >> 16) & 0xffu;
        float tl, tr;
        const bool gl = box_geom(L, o, inv_dir, nx, ny, nz, &tl);
        const bool gr = box_geom(R, o, inv_dir, nx, ny, nz, &tr);
        const bool neg = sc.dist_order ? (tr < tl) : (axis == 0 ? nx : (axis == 1 ? ny : nz));
        const bool gn = neg ? gr : gl, gf = neg ? gl : gr;
        const float tn = neg ? tr : tl, tf = neg ? tl : tr;
        const float4 nb = neg ? R.b : L.b, fb = neg ? L.b : R.b;
        ++*c_nodes;  // the near child's test; the far child's is counted when it is popped
        if (sp_ < PT_STACK_SIZE) stack[sp_] = make_uint4(__float_as_uint(gf ? tf : CUDART_INF_F), __float_as_uint(fb.z), __float_as_uint(fb.w), 0u);
        ++sp_;
        if (gn && tn < t_max) {
          cur_off = __float_as_uint(nb.z);
          cur_meta = __float_as_uint(nb.w);
        } else {
          cur_meta = PT_NO_NODE;
        }
      }
    }
    // phase B: triangles of the leaf in hand
    {
      const bool have_leaf = active && !done_ray && cur_meta != PT_NO_NODE && (cur_meta & 0xffffu) != 0;
      uint32_t cnt = have_leaf ? (cur_meta & 0xffffu) : 0u;
      for (uint32_t i = 0; __ballot_sync(FULL, i < cnt) != 0; ++i) {
        if (i < cnt) {
          const uint32_t prim = cur_off + i;
          const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim);
          const float4 v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1);
          const float4 v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
          ++*c_tris;
          float t, b0, b1, b2;
          if (tri_core(mk3(v0), mk3(v1), mk3(v2), o, rp, t_max, &t, &b0, &b1, &b2) &&
              !tri_post_reject(sc, (int)prim, mk3(v0), mk3(v1), mk3(v2), __float_as_uint(v2.w), b0, b1, b2, !any_hit)) {
            found = true;
            hit.prim = (int)prim;
            hit.t = t;
            hit.b0 = b0;
            hit.b1 = b1;
            hit.b2 = b2;
            t_max = t;
            if (any_hit) {
              cnt = 0;
              done_ray = true;
            }
          }
        }
      }
      if (have_leaf) cur_meta = PT_NO_NODE;
    }
    if (active && (done_ray || (cur_meta == PT_NO_NODE && sp_ == 0))) {
      LaneRay r;
      if (work.end(item, hit, found, &r)) start_ray(r);
      else active = false;
    }
  }
}

// ---- any-hit walk over the occlusion tree ----------------------------------------------------------------
// An any-hit ray keeps its t_max until the first hit ends it, so the reference's walk (accelerator.rs:431-475) tests a
// triangle exactly when the slab test of every box on the way to its leaf passes, in whatever order.  Every interior box of
// the reference-built tree contains its children's boxes (ptrs_scene_create checks it before it builds this tree), and
// with nested boxes the slab test of the inner box passing implies that of the outer one (float subtraction and
// multiplication are monotonic; tests/test_occlusion_tree.py sweeps the NaN / infinity / signed-zero cases of box_geom).
// So a triangle is tested iff its own leaf's box passes, and any tree whose child slots hold reference boxes, with the
// reference's leaves under their own boxes, gives the reference's occlusion answer bit for bit in any visit order.
//
// The occlusion tree is that: every 128-byte wide node holds up to four reference nodes (a node and the interior
// descendants the collapse replaced are skipped: their boxes contain the ones tested below them).  Layout, by plane:
//   float4 [0..6)  min.x, max.x, min.y, max.y, min.z, max.z of the four slots
//   float4 [6]     four child words: bit 31 clear = wide node index; set = leaf, (n_prims - 1) << 27 | first primitive;
//                  PT_W_NONE = empty slot (its box is empty, and the word is checked as well)
//   float4 [7]     unused
// Stack entries are child words: 4 bytes, no entry distance (nothing is re-tested at pop time, t_max does not change).
#define PT_W_NONE 0xffffffffu
#define PT_W_LEAF_BIT 0x80000000u
#define PT_W_IS_LEAF(w) (((w) & PT_W_LEAF_BIT) != 0u && (w) != PT_W_NONE)
#define PT_W_IS_INTERIOR(w) (((w) & PT_W_LEAF_BIT) == 0u)
#define PT_W_LEAF_OFF(w) ((w) & 0x07ffffffu)
#define PT_W_LEAF_CNT(w) ((((w) >> 27) & 15u) + 1u)
// up to three entries per wide level (a node's fourth entered child is the next node in hand); the wide tree is no deeper
// than the reference's, which ptrs_scene_create limits to 64 levels
#define PT_OSTACK_SIZE (3 * PT_STACK_SIZE)

// Warp refill, box phase with one parked leaf, triangle phase: trace_fast's scheme without ordering obligations.
// Work as for trace_fast; every ray is traced as an any-hit ray.
template <class Work>
PT_DEV void trace_occlusion(const DevScene& sc, uint32_t n_items, uint32_t* ticket, Work& work) {
  if (sc.n_wnodes == 0) {
    trace_empty(n_items, ticket, work);
    return;
  }
  const uint32_t FULL = 0xffffffffu;
  const int box_min = (int)sc.box_min;
  uint32_t stack[PT_OSTACK_SIZE];
  int sp_ = 0;
  uint32_t cur = PT_W_NONE;         // entry in hand: wide node, leaf, or none
  uint32_t pl_off = 0, pl_cnt = 0;  // parked leaf: next primitive, triangles left (0 = none)
  uint32_t rbits = 0;               // PT_RB_LIVE, kz
  bool exhausted = n_items == 0;
  uint32_t item = 0;
  V3 o = mk3(0, 0, 0), inv_dir = mk3(0, 0, 0);
  float sx = 0.f, sy = 0.f, sz = 0.f;
  float t_max = 0.f;
  int hit_prim = -1;

  auto start_ray = [&](const LaneRay& r) {
    o = r.o;
    inv_dir = mk3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z);
    const RayPre rp = ray_precompute(r.d);
    sx = rp.sx;
    sy = rp.sy;
    sz = rp.sz;
    rbits = PT_RB_LIVE | ((uint32_t)rp.kz << PT_RB_KZ_SHIFT);
    t_max = r.t_max;
    hit_prim = -1;
    sp_ = 0;
    pl_cnt = 0;
    cur = 0u;  // the root's own box is not tested: it contains every leaf box
  };

  for (;;) {
    // ---- refill ------------------------------------------------------------------------------------
    const uint32_t idle = __ballot_sync(FULL, !(rbits & PT_RB_LIVE));
    if (!exhausted && (__popc(idle) >= PT_REFILL_IDLE)) {
      const int lane = threadIdx.x & 31;
      const int leader = __ffs(idle) - 1;
      uint32_t base = 0;
      if (lane == leader) base = atomicAdd(ticket, (uint32_t)__popc(idle));
      base = __shfl_sync(FULL, base, leader);
      if (base + (uint32_t)__popc(idle) >= n_items) exhausted = true;
      if (!(rbits & PT_RB_LIVE)) {
        const uint32_t i = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
        if (i < n_items) {
          LaneRay r;
          if (work.begin(i, &r)) {
            item = i;
            start_ray(r);
          }
        }
      }
    }
    if (__ballot_sync(FULL, rbits & PT_RB_LIVE) == 0) {
      if (exhausted) break;
      continue;
    }

    // ---- box phase ------------------------------------------------------------------------------------
    // (a lane without a ray has no entry in hand, an empty stack and no parked leaf)
    auto box_step = [&]() {
      if (cur == PT_W_NONE && sp_ > 0) cur = stack[--sp_];
      if (PT_W_IS_LEAF(cur) && pl_cnt == 0u) {
        pl_off = PT_W_LEAF_OFF(cur);
        pl_cnt = PT_W_LEAF_CNT(cur);
        cur = PT_W_NONE;
      }
      if (!PT_W_IS_INTERIOR(cur)) return;
      const float4* nd = sc.wnodes + 8 * (size_t)cur;
      const float4 lx = __ldg(nd), hx = __ldg(nd + 1), ly = __ldg(nd + 2), hy = __ldg(nd + 3), lz = __ldg(nd + 4), hz = __ldg(nd + 5);
      const uint4 ch = __ldg(reinterpret_cast<const uint4*>(nd + 6));
      const bool nx = inv_dir.x < 0.0f, ny = inv_dir.y < 0.0f, nz = inv_dir.z < 0.0f;
      cur = PT_W_NONE;
      auto child = [&](float x0, float x1, float y0, float y1, float z0, float z1, uint32_t w) {
        NodeLoad n;
        n.a = make_float4(x0, y0, z0, x1);
        n.b = make_float4(y1, z1, 0.f, 0.f);
        float te;
        if (box_geom(n, o, inv_dir, nx, ny, nz, &te) && te < t_max && w != PT_W_NONE) {
          if (PT_W_IS_LEAF(w) && pl_cnt == 0u) {
            pl_off = PT_W_LEAF_OFF(w);
            pl_cnt = PT_W_LEAF_CNT(w);
          } else if (cur == PT_W_NONE) {
            cur = w;
          } else if (sp_ < PT_OSTACK_SIZE) {  // always true, see PT_OSTACK_SIZE
            stack[sp_++] = w;
          }
        }
      };
      child(lx.x, hx.x, ly.x, hy.x, lz.x, hz.x, ch.x);
      child(lx.y, hx.y, ly.y, hy.y, lz.y, hz.y, ch.y);
      child(lx.z, hx.z, ly.z, hy.z, lz.z, hz.z, ch.z);
      child(lx.w, hx.w, ly.w, hy.w, lz.w, hz.w, ch.w);
    };
    for (;;) {
      const bool live = (rbits & PT_RB_LIVE) != 0;
      const bool can_box = PT_W_IS_INTERIOR(cur) || (cur == PT_W_NONE && sp_ > 0) || (PT_W_IS_LEAF(cur) && pl_cnt == 0u);
      const uint32_t bmask = __ballot_sync(FULL, can_box);
      if (bmask == 0) break;
      if (__popc(bmask) < box_min && __ballot_sync(FULL, live && !can_box) != 0) break;
#pragma unroll
      for (int rep = 0; rep < PT_BOX_STEPS; ++rep) box_step();
    }

    // ---- triangle phase: the parked leaf, then the leaf in hand ---------------------------------------
    auto tri_step = [&]() {
      if (pl_cnt == 0u && PT_W_IS_LEAF(cur)) {
        pl_off = PT_W_LEAF_OFF(cur);
        pl_cnt = PT_W_LEAF_CNT(cur);
        cur = PT_W_NONE;
      }
      if (pl_cnt != 0u) {
        const uint32_t prim = pl_off;
        const float4 v0 = __ldg(sc.tri_verts + 3 * (size_t)prim);
        const float4 v1 = __ldg(sc.tri_verts + 3 * (size_t)prim + 1);
        const float4 v2 = __ldg(sc.tri_verts + 3 * (size_t)prim + 2);
        ++pl_off;
        --pl_cnt;
        RayPre rp;
        rp.kz = (int)((rbits >> PT_RB_KZ_SHIFT) & 3u);
        rp.sx = sx;
        rp.sy = sy;
        rp.sz = sz;
        float t, b0, b1, b2;
        if (tri_core(mk3(v0), mk3(v1), mk3(v2), o, rp, t_max, &t, &b0, &b1, &b2) &&
            !tri_post_reject(sc, (int)prim, mk3(v0), mk3(v1), mk3(v2), __float_as_uint(v2.w), b0, b1, b2, false)) {
          hit_prim = (int)prim;  // intersect_p returns at the first hit (accelerator.rs:435-442)
          pl_cnt = 0;
          sp_ = 0;
          cur = PT_W_NONE;
        }
      }
    };
    for (;;) {
      const bool has = pl_cnt != 0u || PT_W_IS_LEAF(cur);
      if (__ballot_sync(FULL, has) == 0) break;
      tri_step();
    }

    // ---- rays that ran out of nodes --------------------------------------------------------------------
    if ((rbits & PT_RB_LIVE) && cur == PT_W_NONE && sp_ == 0 && pl_cnt == 0u) {
      DevHit h;
      h.prim = hit_prim;
      h.t = t_max;
      h.b0 = h.b1 = h.b2 = 0.f;
      LaneRay r;
      if (work.end(item, h, hit_prim >= 0, &r)) start_ray(r);
      else rbits = 0;
    }
  }
}

template <bool COUNT, bool DIST, class Work>
PT_DEV void trace_stream(const DevScene& sc, uint32_t n_items, uint32_t* ticket, Work& work, uint32_t* c_nodes, uint32_t* c_tris) {
  if (COUNT) trace_counted(sc, n_items, ticket, work, c_nodes, c_tris);  // (reads sc.dist_order at run time)
  else trace_fast<DIST>(sc, n_items, ticket, work);
}

}  // namespace ptrs
