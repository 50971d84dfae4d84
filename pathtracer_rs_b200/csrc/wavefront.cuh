// Wavefront path-tracing kernels for sm_100a: generate / extend / shade<material> / connect /
// accumulate, plus the standalone closest-hit / any-hit kernels behind ptrs_intersect*.
//
// Execution model
//   * every kernel is persistent: grid = k x 148 SMs, each warp pulls 32 work items at a time from
//     a device-side ticket with ONE atomicAdd per warp (warp-aggregated fetch) until the queue whose
//     length sits in device memory is drained — no host round trip between bounces
//   * queues hold path-slot indices; extend classifies hits by material type and appends to one
//     queue per material class with ballot-aggregated atomics (one atomic per class per warp), so
//     every shade<MAT> launch runs warps that are uniform in material code (material sorting)
//   * shade emits at most three rays per path and bounce — the extension ray into the next round's
//     extend queue, the NEE shadow segment and the MIS ray as one direct-lighting record in the connect
//     queue plus one q_ray entry per ray that exists
//   * connect traces the listed shadow (any-hit) and MIS (closest-hit) rays, one ray per work item;
//     connect_resolve then adds beta * n_lights * (Ld_light + Ld_bsdf) to the path's radiance, one thread
//     per record: a single writer per path per launch keeps the float summation order of
//     integrator.rs:443-447
//   * per-round counters (queue lengths, tickets) live in one zero-initialised block per batch
//
// Path state: 64-byte slot records + queue-ordered payloads, see PathArrays below.
#pragma once
#include <cstddef>
#include "dev_shading.cuh"
#include "dev_sobol.cuh"

namespace ptrs {

#define PT_N_CLASSES (PTRS_MAT_COUNT + 1)  // material types + "miss"
#define PT_CLASS_MISS PTRS_MAT_COUNT

// ---- path state ---------------------------------------------------------------------------------------
// Per path SLOT (indexed by p, gathered): one 64-byte, 64-byte-aligned record read / written with 256-bit
// accesses, so a gather touches whole 32-byte sectors only.
//   [0,32)   next ray + the words every bounce rewrites   (extend reads just this half)
//   [32,64)  throughput + per-path constants
// Per QUEUE ENTRY (indexed by queue position, coalesced): the producer's payload for the consumer —
//   class queues   q_class[i] = slot, q_hit[i] = (primitive, b0, b1, b2)        extend -> shade
//   connect queue  q_nee[i]   = slot, nee[i]   = 96-byte direct-lighting record  shade  -> connect
// Radiance L is a separate float4 per slot: only connect (every bounce), shade (emitters) and
// shade_miss touch it.
struct __align__(32) PathRay {
  float ox, oy, oz;
  uint32_t packed;  // bits 0..15 Sobol dimension, PT_F_* (bits 16, 17), bits 24..31 bounces (signed 8 bit)
  float dx, dy, dz;
  float eta_scale;
};
struct __align__(32) PathAux {
  float br, bg, bb;  // beta
  uint32_t pixel;    // x | y << 16, two int16 (sample-bounds coordinates)
  uint32_t sample;   // sample number of the pixel (Sobol frame)
  uint32_t spare;
  float fx, fy;  // p_film
};
struct __align__(64) PathSlot {
  PathRay r;
  PathAux a;
};
struct __align__(32) NeeRec {  // pending direct-lighting record of the current bounce (estimate_direct, integrator.rs:23-139)
  float4 n0;  // shadow origin xyz,            A.r   (A = f * Li * w / light_pdf)
  float4 n1;  // shadow segment xyz,           A.g
  float4 n2;  // MIS ray origin xyz,           A.b
  float4 n3;  // MIS ray dir xyz,              bits: light id | PT_NEE_*
  float4 n4;  // f (already * |wi.ns|) rgb,     MIS weight
  float4 n5;  // beta before the bounce rgb,   scattering pdf
};
struct __align__(32) NeeRes {  // what connect_trace found for NeeRec i
  int prim;  // MIS ray: closest primitive or -1
  float b0, b1, b2;
  uint32_t occluded;  // shadow segment blocked
  uint32_t pad[3];
};
struct PathArrays {
  PathSlot* slot;
  float4* L;        // rgb
  float4* q_hit;    // PT_N_CLASSES x cap, aligned with the class queues
  NeeRec* nee;      // cap, aligned with the connect queue
  NeeRes* nee_res;  // cap, aligned with the connect queue
  uint32_t* q_ray;  // 2 x cap: the rays the connect stage has to trace, 2 * record + {0 shadow segment, 1 MIS ray} (RoundCounters)
};
#define PT_F_SPECULAR (1u << 16)
#define PT_F_HAS_DIFF (1u << 17)
#define PT_NEE_SHADOW (1u << 30)
#define PT_NEE_MIS (1u << 31)
// The MIS ray of an INFINITE light only asks whether it escapes: estimate_direct (integrator.rs:113-135) adds
// light.le(ray) when scene.intersect finds nothing and, when it finds something, compares the hit primitive's area light
// with the sampled light — which an infinite light never is.  scene.intersect(ray) and scene.intersect_p(ray) agree on
// "something is hit" (same triangle test; the closest-hit path's extra rejection of degenerate partials is unreachable,
// a zero-area triangle fails det != 0 first), so such a ray is traced as an any-hit ray and stops at the first hit.
#define PT_NEE_MIS_ANY (1u << 29)
#define PT_NEE_LIGHT_MASK 0x1fffffffu
PT_DEV uint32_t pack_state(uint32_t dim_and_flags, int bounces) { return (dim_and_flags & 0x00ffffffu) | ((uint32_t)(bounces & 0xff) << 24); }
PT_DEV int packed_bounces(uint32_t packed) { return (int)(int8_t)(packed >> 24); }
PT_DEV uint32_t pack_pixel(int x, int y) { return ((uint32_t)x & 0xffffu) | ((uint32_t)y << 16); }
PT_DEV int2 unpack_pixel(uint32_t v) { return make_int2((int)(int16_t)(v & 0xffffu), (int)(int16_t)(v >> 16)); }

// 256-bit accesses (LDG.E.256 / STG.E.256, sm_100a)
template <class T>
PT_DEV T ld256(const T* p) {
  static_assert(sizeof(T) == 32, "32-byte record");
  union {
    T v;
    uint32_t w[8];
  } u;
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(u.w[0]), "=r"(u.w[1]), "=r"(u.w[2]), "=r"(u.w[3]), "=r"(u.w[4]), "=r"(u.w[5]), "=r"(u.w[6]), "=r"(u.w[7])
               : "l"(p)
               : "memory");
  return u.v;
}
template <class T>
PT_DEV void st256(T* p, const T& v) {
  static_assert(sizeof(T) == 32, "32-byte record");
  union {
    T v;
    uint32_t w[8];
  } u;
  u.v = v;
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(u.w[0]), "r"(u.w[1]), "r"(u.w[2]), "r"(u.w[3]), "r"(u.w[4]), "r"(u.w[5]),
               "r"(u.w[6]), "r"(u.w[7])
               : "memory");
}
struct __align__(32) F8 {
  float4 a, b;
};
PT_DEV void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
PT_DEV void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// per-round device counters; one RoundCounters per extend/shade/connect round of a batch
struct RoundCounters {
  uint32_t n_ext;                  // length of the extend queue of this round
  uint32_t n_class[PT_N_CLASSES];  // lengths of the per-material shade queues
  // connect stage: direct-lighting records and the rays of those records (q_ray).  The pair is one 8-byte
  // aligned word so that shade reserves both with a single 64-bit atomicAdd (records in the low half).
  // n_ray counts the any-hit rays at the bottom of q_ray, n_ray_closest the closest-hit MIS rays at its top
  // (q_ray[2 * cap - 1 - j]); the two never meet, every record has at most two rays
  uint32_t n_nee, n_ray;
  uint32_t t_ext, t_class[PT_N_CLASSES], t_nee, t_ray;  // work tickets
  uint32_t n_ray_closest, t_ray_closest;
  uint32_t pad[32 - 8 - 2 * PT_N_CLASSES];  // 128 B per round
};
static_assert(offsetof(RoundCounters, n_nee) % 8 == 0 && sizeof(RoundCounters) == 128, "RoundCounters layout");

struct GlobalCounters {
  unsigned long long shadow_rays, mis_rays, nodes_tested, tris_tested, nee_nodes_tested, nee_tris_tested;
};

struct RenderConst {
  SobolConfig sobol;
  SobolSplit split;
  PtrsCamera cam;
  float filter_table[256];
  float filter_radius[2];
  float inv_filter_radius[2];
  float diff_scale;  // 1 / sqrt(spp)
  int32_t max_depth;
  float rr_threshold;
  int32_t rr_start_depth;
  int32_t rr_enable;
  int32_t sb_min[2], sb_ext[2];  // sample bounds min and extent
  // the rectangle of sample positions the generate kernel enumerates: the sample bounds or a sub-rectangle of them
  // (ptrs_render_region).  The Sobol index and the split tables stay relative to the full sample bounds.
  int32_t rect_min[2], rect_ext[2];
  int32_t s_begin, s_count, s_stride, s_phase;  // sample numbers: s = s_begin + s_phase' + j * s_stride
  uint32_t cap;
};

// ---- work fetch --------------------------------------------------------------------------------------
PT_DEV uint32_t warp_fetch32(uint32_t* ticket) {
  uint32_t base = 0;
  if ((threadIdx.x & 31) == 0) base = atomicAdd(ticket, 32u);
  return __shfl_sync(0xffffffffu, base, 0);
}
// append `item` for lanes with pred to queue q (length counter n) — one atomic per warp
PT_DEV void warp_push(bool pred, uint32_t item, int* q, uint32_t* n) {
  const uint32_t mask = __ballot_sync(0xffffffffu, pred);
  if (mask == 0) return;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(mask) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(n, (uint32_t)__popc(mask));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (pred) q[base + __popc(mask & ((1u << lane) - 1))] = (int)item;
}
PT_DEV void warp_count(bool pred, unsigned long long* ctr) {
  const uint32_t mask = __ballot_sync(0xffffffffu, pred);
  if (mask && (threadIdx.x & 31) == (__ffs(mask) - 1)) atomicAdd(ctr, (unsigned long long)__popc(mask));
}
PT_DEV void warp_sum_add(uint32_t v, unsigned long long* ctr) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(ctr, (unsigned long long)v);
}

// ---- camera ----------------------------------------------------------------------------------------
PT_DEV V3 quat_rotate(const float q[4], V3 v) {  // UnitQuaternion * Vector3 (nalgebra)
  V3 qv = mk3(q[0], q[1], q[2]);
  V3 t = cross(qv, v) * 2.0f;
  V3 c = cross(qv, t);
  return t * q[3] + c + v;
}
// Camera::generate_ray_differential + scale_differentials (pathtracer/mod.rs:59-81, ray.rs:30-35)
PT_DEV void camera_ray(const PtrsCamera& cam, float fx, float fy, float diff_scale, V3* o, V3* d, V3* rx_d, V3* ry_d) {
  const float* m = cam.raster_to_screen;
  float sx = (m[0] * fx + m[1] * fy) + m[2] * 0.0f + m[3];
  float sy = (m[4] * fx + m[5] * fy) + m[6] * 0.0f + m[7];
  float sz = (m[8] * fx + m[9] * fy) + m[10] * 0.0f + m[11];
  float inverse_denom = cam.persp[3] / (sz + cam.persp[2]);
  V3 pc = mk3(sx * inverse_denom / cam.persp[0], sy * inverse_denom / cam.persp[1], -inverse_denom);
  *o = mk3(cam.trans[0], cam.trans[1], cam.trans[2]);
  *d = normalize(quat_rotate(cam.rot, pc));
  if (rx_d) {
    V3 rx = normalize(quat_rotate(cam.rot, pc + mk3(cam.dx_camera[0], cam.dx_camera[1], cam.dx_camera[2])));
    V3 ry = normalize(quat_rotate(cam.rot, pc + mk3(cam.dy_camera[0], cam.dy_camera[1], cam.dy_camera[2])));
    *rx_d = *d + (rx - *d) * diff_scale;
    *ry_d = *d + (ry - *d) * diff_scale;
  }
}

}  // namespace ptrs
