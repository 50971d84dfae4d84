// The reference's binned SAH build (BVH::new, src/pathtracer/accelerator.rs:103-346) on the device, bit for bit: the
// records and the primitive order equal ptrs_host::build_bvh(bounds, max_prims, 1) (host/bvh_build.cpp, the spec every
// "bvh_build.cpp:N" below cites), so a scene built from them is the ptrs_scene_create scene of the same primitives.
//
// Schedule.  Nodes of more than SAH_SMALL primitives are built level by level over the whole primitive array: a node box
// and centroid-bounds reduction, one thread per node to pick the axis, a bucket pass, one thread per node for the 11
// costs, and the partition as a scan + pair + swap.  One read-back per level (counters).  A node of at most SAH_SMALL
// primitives is a subtree one thread finishes with the host recursion written out (build_small).  The finished BFS
// topology becomes the reference's depth-first preorder: subtree sizes bottom-up, preorder indices top-down, emission.
//
// Where a parallel build could diverge from the host's, and what keeps it equal:
//  * fmin / fmax: std::fmin ignores NaN and returns its FIRST argument on ties (fmin(+0, -0) = +0, fmin(-0, +0) = -0).
//    h_fmin / h_fmax restate that rule.  A node's box is a left fold from +-FLT_MAX in the node's current array order:
//    the min over non-NaN values, clamped to FLT_MAX, with the sign of a zero from the lowest position.  The level pass
//    reduces (value with -0 == +0, position) keys and then reads the winner's value, which gives exactly that.
//  * Bucket boxes and centroid bounds feed only comparisons, differences that are compared, and surface areas whose
//    zero sign cannot change a cost (1 + (+-0) / sa == 1 + 0 / sa, and 0 / 0 is NaN either way).  Order-preserving integer
//    atomics that skip NaN, from +-FLT_MAX, give their values up to the sign of a zero.
//  * partition_in_place swaps the k-th "false" from the left with the k-th "true" from the right: with c trues, the
//    falses in [start, start + c) pair with the trues in [start + c, end) by rank, from one scan of the flags.
#include <cfloat>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>
#include <cub/device/device_scan.cuh>

#include "launch.hpp"

namespace ptrs {

namespace {

constexpr int SAH_BUCKETS = 12;        // bvh_build.cpp:60
constexpr uint32_t SAH_SMALL = 128;    // nodes of at most this many primitives: one thread builds the subtree
constexpr uint32_t SAH_NONE = 0xffffffffu;
constexpr int SAH_TILE_ITEMS = 8;
constexpr uint32_t SAH_TILE = 256 * SAH_TILE_ITEMS;

struct Bounds {
  float mn[3], mx[3];
};
struct Prim {  // PrimInfo, bvh_build.cpp:54-58
  float mn[3], mx[3], c[3];
  uint32_t id;
};

// std::fmin / std::fmax as glibc computes them: the second argument only when it is smaller (larger) or the first is NaN
__device__ __forceinline__ float h_fmin(float x, float y) { return (y < x || x != x) ? y : x; }
__device__ __forceinline__ float h_fmax(float x, float y) { return (y > x || x != x) ? y : x; }

__device__ __forceinline__ Bounds empty_bounds() { return Bounds{{FLT_MAX, FLT_MAX, FLT_MAX}, {-FLT_MAX, -FLT_MAX, -FLT_MAX}}; }  // :14-16
__device__ __forceinline__ void bunion(Bounds& r, const float mn[3], const float mx[3]) {  // :18-25
  for (int k = 0; k < 3; ++k) {
    r.mn[k] = h_fmin(r.mn[k], mn[k]);
    r.mx[k] = h_fmax(r.mx[k], mx[k]);
  }
}
__device__ __forceinline__ float surface_area(const Bounds& b) {  // :35-38
  float dx = b.mx[0] - b.mn[0], dy = b.mx[1] - b.mn[1], dz = b.mx[2] - b.mn[2];
  return 2.0f * (dx * dy + dx * dz + dy * dz);
}
__device__ __forceinline__ int maximum_extent(const Bounds& b) {  // :40-46
  float d[3] = {b.mx[0] - b.mn[0], b.mx[1] - b.mn[1], b.mx[2] - b.mn[2]};
  int best = 0;
  for (int k = 1; k < 3; ++k)
    if (d[k] > d[best]) best = k;
  return best;
}
// bucket_of (:48-52 and :62-68) on the split axis only: cmn / cmx are the centroid bounds on `dim`
__device__ __forceinline__ int bucket_of(float cmn, float cmx, float p) {
  float o = p - cmn;
  if (cmx > cmn) o /= cmx - cmn;
  float f = (float)SAH_BUCKETS * o;
  if (!(f > 0.0f)) return 0;
  if (f >= (float)SAH_BUCKETS) return SAH_BUCKETS - 1;
  return (int)f;
}
// :124-145, verbatim: the 11 split costs and the first minimum by strict <
__device__ __forceinline__ void split_costs(const uint32_t count[SAH_BUCKETS], const Bounds bb[SAH_BUCKETS], const Bounds& bounds, float* min_cost_out,
                                            int* split_out) {
  float cost[SAH_BUCKETS - 1];
  const float inv_total_sa_den = surface_area(bounds);
  for (int i = 0; i < SAH_BUCKETS - 1; ++i) {
    Bounds b0 = empty_bounds(), b1 = empty_bounds();
    uint64_t c0 = 0, c1 = 0;
    for (int j = 0; j <= i; ++j) {
      bunion(b0, bb[j].mn, bb[j].mx);
      c0 += count[j];
    }
    for (int j = i + 1; j < SAH_BUCKETS; ++j) {
      bunion(b1, bb[j].mn, bb[j].mx);
      c1 += count[j];
    }
    cost[i] = 1.0f + ((float)c0 * surface_area(b0) + (float)c1 * surface_area(b1)) / inv_total_sa_den;
  }
  float min_cost = cost[0];
  int split = 0;
  for (int i = 1; i < SAH_BUCKETS - 1; ++i)
    if (cost[i] < min_cost) {
      min_cost = cost[i];
      split = i;
    }
  *min_cost_out = min_cost;
  *split_out = split;
}

// order-preserving float <-> uint map (k_bvh.cu's f2o / o2f)
__device__ __forceinline__ uint32_t f2o(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float o2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }
// (value, position) keys of the node-box fold: -0 and +0 share a value, so the lower position decides between them
__device__ __forceinline__ unsigned long long key_min(float v, uint32_t pos) { return ((unsigned long long)f2o(v == 0.0f ? 0.0f : v) << 32) | pos; }
__device__ __forceinline__ unsigned long long key_max(float v, uint32_t pos) { return ((unsigned long long)f2o(v == 0.0f ? 0.0f : v) << 32) | (uint32_t)~pos; }

// one 32-byte LinearBVHNode record as two float4 (PtrsBvhNode: bounds, offset, n_prims, axis, pad = 0)
__device__ __forceinline__ void put_record(float4* out, const Bounds& b, uint32_t offset, uint32_t n_prims, uint32_t axis) {
  out[0] = make_float4(b.mn[0], b.mn[1], b.mn[2], b.mx[0]);
  out[1] = make_float4(b.mx[1], b.mx[2], __uint_as_float(offset), __uint_as_float(n_prims | (axis << 16)));
}

enum : uint32_t { SAH_INTERIOR = 0, SAH_LEAF = 1, SAH_SUBTREE = 2, SAH_PENDING = 3 };
struct SahNode {  // one node of the level phase, by BFS id
  Bounds box;
  uint32_t start, end;
  uint32_t child;  // SAH_INTERIOR: BFS id of the first child (the second is child + 1); SAH_SUBTREE: index in the subtree list
  uint32_t depth;  // 1 at the root, as bvh_build.cpp counts it
  uint32_t kind, dim;
};
struct SegAcc {  // reductions of one node of the current level
  unsigned long long kmin[3], kmax[3];
  uint32_t cmin[3], cmax[3];
  uint32_t cnt[SAH_BUCKETS];
  uint32_t bmin[SAH_BUCKETS][3], bmax[SAH_BUCKETS][3];
};
enum : uint32_t { PLAN_DONE = 0, PLAN_BUCKETS = 1, PLAN_PARTITION = 2, PLAN_HALVE = 3 };
struct SegPlan {
  uint32_t node, mode, split, mid;
  uint32_t next[2];  // slots of the two children on the next level (SAH_NONE: a subtree or nothing)
  float cmn, cmx;    // centroid bounds on dim
  uint32_t dim;
};
struct Counters {
  uint32_t n_bfs, n_next, n_sub, max_depth;
};

__global__ void __launch_bounds__(256) sah_prims_kernel(uint32_t n, const uint32_t* __restrict__ prim_vertex, const float* __restrict__ pos, Prim* __restrict__ P) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
    Prim p;
    for (int k = 0; k < 3; ++k) {  // Triangle::world_bound as SceneBuilder::finalize computes it (scene_builder.cpp:472-481)
      const float a = pos[3 * (size_t)prim_vertex[3 * (size_t)t] + k], c = pos[3 * (size_t)prim_vertex[3 * (size_t)t + 1] + k],
                  d = pos[3 * (size_t)prim_vertex[3 * (size_t)t + 2] + k];
      p.mn[k] = h_fmin(h_fmin(a, c), d);
      p.mx[k] = h_fmax(h_fmax(a, c), d);
    }
    for (int k = 0; k < 3; ++k) p.c[k] = p.mn[k] + 0.5f * (p.mx[k] - p.mn[k]);  // bvh_build.cpp:220-221
    p.id = t;
    P[t] = p;
  }
}

__global__ void sah_acc_init_kernel(uint32_t n_active, SegAcc* __restrict__ acc) {
  const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_active) return;
  SegAcc& A = acc[a];
  for (int k = 0; k < 3; ++k) {
    A.kmin[k] = ~0ull;
    A.kmax[k] = 0ull;
    A.cmin[k] = f2o(FLT_MAX);
    A.cmax[k] = f2o(-FLT_MAX);
  }
  for (int b = 0; b < SAH_BUCKETS; ++b) {
    A.cnt[b] = 0;
    for (int k = 0; k < 3; ++k) {
      A.bmin[b][k] = f2o(FLT_MAX);
      A.bmax[b][k] = f2o(-FLT_MAX);
    }
  }
}

// node boxes (exact fold keys) and centroid bounds.  Every thread keeps its own reduction for the node of its tile's
// first element; a warp combines them with shuffles and one lane goes to global memory.  Elements of other nodes
// (small ones, at a tile's end) go to global memory directly.
__global__ void __launch_bounds__(256) sah_box_kernel(uint32_t n, const Prim* __restrict__ P, const uint32_t* __restrict__ seg, SegAcc* __restrict__ acc) {
  const uint32_t lane = threadIdx.x & 31;
  for (uint32_t base = blockIdx.x * SAH_TILE; base < n; base += gridDim.x * SAH_TILE) {
    const uint32_t s0 = seg[base];
    unsigned long long kmin[3] = {~0ull, ~0ull, ~0ull}, kmax[3] = {0ull, 0ull, 0ull};
    uint32_t cmin[3] = {SAH_NONE, SAH_NONE, SAH_NONE}, cmax[3] = {0u, 0u, 0u};
    for (int j = 0; j < SAH_TILE_ITEMS; ++j) {
      const uint32_t i = base + j * 256 + threadIdx.x;
      if (i >= n) break;
      const uint32_t s = seg[i];
      if (s == SAH_NONE) continue;
      const Prim& p = P[i];
      for (int k = 0; k < 3; ++k) {
        const float lo = p.mn[k], hi = p.mx[k], c = p.c[k];
        if (s == s0) {
          if (lo == lo) kmin[k] = min(kmin[k], key_min(lo, i));
          if (hi == hi) kmax[k] = max(kmax[k], key_max(hi, i));
          if (c == c) {
            cmin[k] = min(cmin[k], f2o(c));
            cmax[k] = max(cmax[k], f2o(c));
          }
        } else {
          SegAcc& A = acc[s];
          if (lo == lo) atomicMin(&A.kmin[k], key_min(lo, i));
          if (hi == hi) atomicMax(&A.kmax[k], key_max(hi, i));
          if (c == c) {
            atomicMin(&A.cmin[k], f2o(c));
            atomicMax(&A.cmax[k], f2o(c));
          }
        }
      }
    }
    if (s0 == SAH_NONE) continue;
    for (int o = 16; o > 0; o >>= 1)
      for (int k = 0; k < 3; ++k) {
        kmin[k] = min(kmin[k], __shfl_xor_sync(0xffffffffu, kmin[k], o));
        kmax[k] = max(kmax[k], __shfl_xor_sync(0xffffffffu, kmax[k], o));
        cmin[k] = min(cmin[k], __shfl_xor_sync(0xffffffffu, cmin[k], o));
        cmax[k] = max(cmax[k], __shfl_xor_sync(0xffffffffu, cmax[k], o));
      }
    if (lane == 0) {
      SegAcc& A = acc[s0];
      for (int k = 0; k < 3; ++k) {
        if (kmin[k] != ~0ull) atomicMin(&A.kmin[k], kmin[k]);
        if (kmax[k] != 0ull) atomicMax(&A.kmax[k], kmax[k]);
        if (cmin[k] != SAH_NONE) atomicMin(&A.cmin[k], cmin[k]);
        if (cmax[k] != 0u) atomicMax(&A.cmax[k], cmax[k]);
      }
    }
  }
}

// children of a node that splits at `mid`: BFS ids, and a slot on the next level or a place in the subtree list
__device__ void sah_split(SahNode* __restrict__ nodes, uint32_t id, uint32_t mid, SegPlan& pl, Counters* ctr, uint32_t* __restrict__ next_active,
                          uint32_t* __restrict__ sub_list) {
  SahNode& nd = nodes[id];
  const uint32_t c = atomicAdd(&ctr->n_bfs, 2u);
  nd.kind = SAH_INTERIOR;
  nd.child = c;
  pl.mid = mid;
  const uint32_t lo[2] = {nd.start, mid}, hi[2] = {mid, nd.end};
  for (int h = 0; h < 2; ++h) {
    SahNode& ch = nodes[c + h];
    ch.start = lo[h];
    ch.end = hi[h];
    ch.depth = nd.depth + 1;
    if (hi[h] - lo[h] > SAH_SMALL) {
      const uint32_t slot = atomicAdd(&ctr->n_next, 1u);
      next_active[slot] = c + h;
      ch.kind = SAH_PENDING;
      pl.next[h] = slot;
    } else {
      const uint32_t k = atomicAdd(&ctr->n_sub, 1u);
      sub_list[k] = c + h;
      ch.kind = SAH_SUBTREE;
      ch.child = k;
      pl.next[h] = SAH_NONE;
    }
  }
  atomicMax(&ctr->max_depth, nd.depth + 1);
}

// one thread per node of the level: its box, the split axis, and the tests that come before the buckets (:96-110)
__global__ void sah_decide_kernel(uint32_t n_active, const uint32_t* __restrict__ active, SahNode* __restrict__ nodes, const Prim* __restrict__ P,
                                  const SegAcc* __restrict__ acc, SegPlan* __restrict__ plan, Counters* ctr, uint32_t* __restrict__ next_active,
                                  uint32_t* __restrict__ sub_list) {
  const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_active) return;
  const uint32_t id = active[a];
  SahNode& nd = nodes[id];
  const SegAcc& A = acc[a];
  Bounds b, cb;
  for (int k = 0; k < 3; ++k) {  // the fold of :82-83: the winning element's own value, clamped to +-FLT_MAX
    const float lo = A.kmin[k] == ~0ull ? FLT_MAX : P[(uint32_t)A.kmin[k]].mn[k];
    const float hi = A.kmax[k] == 0ull ? -FLT_MAX : P[~(uint32_t)A.kmax[k]].mx[k];
    b.mn[k] = lo < FLT_MAX ? lo : FLT_MAX;
    b.mx[k] = hi > -FLT_MAX ? hi : -FLT_MAX;
    cb.mn[k] = o2f(A.cmin[k]);
    cb.mx[k] = o2f(A.cmax[k]);
  }
  nd.box = b;
  const int dim = maximum_extent(cb);  // :100-102
  nd.dim = (uint32_t)dim;
  SegPlan pl;
  pl.node = id;
  pl.dim = (uint32_t)dim;
  pl.cmn = cb.mn[dim];
  pl.cmx = cb.mx[dim];
  pl.split = 0;
  pl.mid = nd.start;
  pl.next[0] = pl.next[1] = SAH_NONE;
  // n > SAH_SMALL here, so neither n == 1 (:96) nor n <= 2 (:110) can occur
  const uint32_t n = nd.end - nd.start;
  if (cb.mx[dim] == cb.mn[dim]) {  // :104-109
    if (n <= 65535) {
      nd.kind = SAH_LEAF;
      pl.mode = PLAN_DONE;
    } else {
      pl.mode = PLAN_HALVE;
      sah_split(nodes, id, nd.start + n / 2, pl, ctr, next_active, sub_list);
    }
  } else {
    pl.mode = PLAN_BUCKETS;
  }
  plan[a] = pl;
}

// bucket counts and boxes (:116-123); per-warp copies in shared memory for the node of the tile's first element
__global__ void __launch_bounds__(256) sah_bucket_kernel(uint32_t n, const Prim* __restrict__ P, const uint32_t* __restrict__ seg, const SegPlan* __restrict__ plan,
                                                         SegAcc* __restrict__ acc) {
  __shared__ uint32_t s_cnt[8][SAH_BUCKETS];
  __shared__ uint32_t s_box[8][SAH_BUCKETS][6];
  const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (uint32_t base = blockIdx.x * SAH_TILE; base < n; base += gridDim.x * SAH_TILE) {
    const uint32_t s0 = seg[base];
    const bool own = s0 != SAH_NONE && plan[s0].mode == PLAN_BUCKETS;
    if (lane < SAH_BUCKETS) {
      s_cnt[w][lane] = 0;
      for (int k = 0; k < 3; ++k) {
        s_box[w][lane][k] = f2o(FLT_MAX);
        s_box[w][lane][3 + k] = f2o(-FLT_MAX);
      }
    }
    __syncwarp();
    for (int j = 0; j < SAH_TILE_ITEMS; ++j) {
      const uint32_t i = base + j * 256 + threadIdx.x;
      if (i >= n) break;
      const uint32_t s = seg[i];
      if (s == SAH_NONE) continue;
      const SegPlan& pl = plan[s];
      if (pl.mode != PLAN_BUCKETS) continue;
      const Prim& p = P[i];
      const int bk = bucket_of(pl.cmn, pl.cmx, p.c[pl.dim]);
      if (s == s0) {
        atomicAdd(&s_cnt[w][bk], 1u);
        for (int k = 0; k < 3; ++k) {
          if (p.mn[k] == p.mn[k]) atomicMin(&s_box[w][bk][k], f2o(p.mn[k]));
          if (p.mx[k] == p.mx[k]) atomicMax(&s_box[w][bk][3 + k], f2o(p.mx[k]));
        }
      } else {
        SegAcc& A = acc[s];
        atomicAdd(&A.cnt[bk], 1u);
        for (int k = 0; k < 3; ++k) {
          if (p.mn[k] == p.mn[k]) atomicMin(&A.bmin[bk][k], f2o(p.mn[k]));
          if (p.mx[k] == p.mx[k]) atomicMax(&A.bmax[bk][k], f2o(p.mx[k]));
        }
      }
    }
    __syncwarp();
    if (own && lane < SAH_BUCKETS && s_cnt[w][lane] != 0) {
      SegAcc& A = acc[s0];
      atomicAdd(&A.cnt[lane], s_cnt[w][lane]);
      for (int k = 0; k < 3; ++k) {
        atomicMin(&A.bmin[lane][k], s_box[w][lane][k]);
        atomicMax(&A.bmax[lane][k], s_box[w][lane][3 + k]);
      }
    }
    __syncwarp();
  }
}

// one thread per node with buckets: the costs, the leaf test (:146-147) and the split position
__global__ void sah_cost_kernel(uint32_t n_active, SahNode* __restrict__ nodes, const SegAcc* __restrict__ acc, SegPlan* __restrict__ plan, int max_prims,
                                Counters* ctr, uint32_t* __restrict__ next_active, uint32_t* __restrict__ sub_list) {
  const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_active) return;
  SegPlan pl = plan[a];
  if (pl.mode != PLAN_BUCKETS) return;
  SahNode& nd = nodes[pl.node];
  const SegAcc& A = acc[a];
  Bounds bb[SAH_BUCKETS];
  uint32_t count[SAH_BUCKETS];
  for (int b = 0; b < SAH_BUCKETS; ++b) {
    count[b] = A.cnt[b];
    for (int k = 0; k < 3; ++k) {
      bb[b].mn[k] = o2f(A.bmin[b][k]);
      bb[b].mx[k] = o2f(A.bmax[b][k]);
    }
  }
  float min_cost;
  int split;
  split_costs(count, bb, nd.box, &min_cost, &split);
  const uint32_t n = nd.end - nd.start;
  if (n > (uint32_t)max_prims || min_cost < (float)(uint64_t)n) {
    uint32_t c = 0;
    for (int b = 0; b <= split; ++b) c += count[b];
    pl.split = (uint32_t)split;
    // c == 0 or c == n: partition_in_place moves nothing, and :170 halves the range
    pl.mode = (c == 0 || c == n) ? PLAN_HALVE : PLAN_PARTITION;
    sah_split(nodes, pl.node, pl.mode == PLAN_HALVE ? nd.start + n / 2 : nd.start + c, pl, ctr, next_active, sub_list);
  } else {
    nd.kind = SAH_LEAF;
    pl.mode = PLAN_DONE;
  }
  plan[a] = pl;
}

__global__ void __launch_bounds__(256) sah_flag_kernel(uint32_t n, const Prim* __restrict__ P, const uint32_t* __restrict__ seg, const SegPlan* __restrict__ plan,
                                                       uint32_t* __restrict__ flag) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = seg[i];
    uint32_t f = 0;
    if (s != SAH_NONE) {
      const SegPlan& pl = plan[s];
      if (pl.mode == PLAN_PARTITION) f = bucket_of(pl.cmn, pl.cmx, P[i].c[pl.dim]) <= (int)pl.split ? 1u : 0u;  // :150
    }
    flag[i] = f;
  }
}

// the trues in [mid, end), by rank from the right
__global__ void __launch_bounds__(256) sah_pair_kernel(uint32_t n, const uint32_t* __restrict__ seg, const SegPlan* __restrict__ plan, const SahNode* __restrict__ nodes,
                                                       const uint32_t* __restrict__ flag, const uint32_t* __restrict__ scan, uint32_t* __restrict__ right) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = seg[i];
    if (s == SAH_NONE || !flag[i]) continue;
    const SegPlan& pl = plan[s];
    if (i < pl.mid) continue;
    const uint32_t start = nodes[pl.node].start;
    const uint32_t c = pl.mid - start;
    right[start + (c - (scan[i] - scan[start]) - 1u)] = i;
  }
}

// the k-th false in [start, mid) swaps with the k-th true from the right; every element learns its next-level slot
__global__ void __launch_bounds__(256) sah_swap_kernel(uint32_t n, Prim* __restrict__ P, const uint32_t* __restrict__ seg, const SegPlan* __restrict__ plan,
                                                       const SahNode* __restrict__ nodes, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ scan,
                                                       const uint32_t* __restrict__ right, uint32_t* __restrict__ seg_next) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = seg[i];
    uint32_t nx = SAH_NONE;
    if (s != SAH_NONE) {
      const SegPlan& pl = plan[s];
      if (pl.mode == PLAN_PARTITION || pl.mode == PLAN_HALVE) nx = pl.next[i < pl.mid ? 0 : 1];
      if (pl.mode == PLAN_PARTITION && i < pl.mid && !flag[i]) {
        const uint32_t start = nodes[pl.node].start;
        const uint32_t j = right[start + ((i - start) - (scan[i] - scan[start]))];
        const Prim t = P[i];
        P[i] = P[j];
        P[j] = t;
      }
    }
    seg_next[i] = nx;
  }
}

// Builder::build (:77-207) for one node of at most SAH_SMALL primitives, serially, with the recursion as an explicit
// stack.  Records go to out[0 ..) in preorder with interior offsets relative to out; returns their number.
__device__ uint32_t build_small(Prim* __restrict__ P, uint32_t start0, uint32_t end0, int max_prims, float4* __restrict__ out, uint32_t depth0,
                                uint32_t* max_depth) {
  struct Task {
    uint32_t start, end, depth, parent;
  };
  Task stack[SAH_SMALL];  // one entry per pending second child: at most the depth of the subtree, at most its size
  int sp = 0;
  Task cur{start0, end0, depth0, SAH_NONE};
  uint32_t cnt = 0, deepest = depth0;
  while (true) {
    const uint32_t start = cur.start, end = cur.end, my = cnt++;
    if (cur.parent != SAH_NONE) {  // :194-197: the second child starts here
      float4 r = out[2 * cur.parent + 1];
      r.z = __uint_as_float(my);
      out[2 * cur.parent + 1] = r;
    }
    deepest = max(deepest, cur.depth);
    Bounds bounds = empty_bounds();
    for (uint32_t i = start; i < end; ++i) bunion(bounds, P[i].mn, P[i].mx);
    const uint32_t n = end - start;
    uint32_t mid = SAH_NONE;
    int dim = 0;
    if (n > 1) {  // n == 1: a leaf (:96-99)
      Bounds cb = empty_bounds();
      for (uint32_t i = start; i < end; ++i) bunion(cb, P[i].c, P[i].c);
      dim = maximum_extent(cb);
      if (cb.mx[dim] == cb.mn[dim]) {
        // equal centroids: a leaf (n <= SAH_SMALL < 65536, :104-108)
      } else if (n <= 2) {  // :110-114
        mid = start + 1;
        if (P[start + 1].c[dim] < P[start].c[dim]) {
          const Prim t = P[start];
          P[start] = P[start + 1];
          P[start + 1] = t;
        }
      } else {
        uint32_t count[SAH_BUCKETS];
        Bounds bb[SAH_BUCKETS];
        for (int b = 0; b < SAH_BUCKETS; ++b) {
          count[b] = 0;
          bb[b] = empty_bounds();
        }
        for (uint32_t i = start; i < end; ++i) {
          const int b = bucket_of(cb.mn[dim], cb.mx[dim], P[i].c[dim]);
          count[b] += 1;
          bunion(bb[b], P[i].mn, P[i].mx);
        }
        float min_cost;
        int split;
        split_costs(count, bb, bounds, &min_cost, &split);
        if (n > (uint32_t)max_prims || min_cost < (float)(uint64_t)n) {
          uint32_t first = start, last = end;  // :148-160
          auto pred = [&](uint32_t i) { return bucket_of(cb.mn[dim], cb.mx[dim], P[i].c[dim]) <= split; };
          while (true) {
            while (first != last && pred(first)) ++first;
            if (first == last) break;
            --last;
            while (first != last && !pred(last)) --last;
            if (first == last) break;
            const Prim t = P[first];
            P[first] = P[last];
            P[last] = t;
            ++first;
          }
          mid = first;
        }
      }
    }
    if (mid == SAH_NONE) {
      put_record(out + 2 * my, bounds, start, n, 0);
      if (sp == 0) break;
      cur = stack[--sp];
      continue;
    }
    if (mid == start || mid == end) mid = start + n / 2;  // :170
    put_record(out + 2 * my, bounds, 0, 0, (uint32_t)dim);  // offset: patched when the second child starts
    stack[sp++] = Task{mid, end, cur.depth + 1, my};
    cur = Task{start, mid, cur.depth + 1, SAH_NONE};
  }
  *max_depth = deepest;
  return cnt;
}

__global__ void __launch_bounds__(128) sah_small_kernel(uint32_t n_sub, const uint32_t* __restrict__ sub_list, const SahNode* __restrict__ nodes, Prim* __restrict__ P,
                                                        int max_prims, float4* __restrict__ scratch, uint32_t* __restrict__ sub_cnt, Counters* ctr) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_sub) return;
  const SahNode& nd = nodes[sub_list[k]];
  uint32_t deepest = 0;
  // a subtree over [start, end) has at most 2 (end - start) - 1 records: [2 start, 2 end) of the scratch array is its own
  sub_cnt[k] = build_small(P, nd.start, nd.end, max_prims, scratch + 4 * (size_t)nd.start, nd.depth, &deepest);
  atomicMax(&ctr->max_depth, deepest);
}

__global__ void __launch_bounds__(256) sah_size_kernel(uint32_t lo, uint32_t hi, const SahNode* __restrict__ nodes, const uint32_t* __restrict__ sub_cnt,
                                                       uint32_t* __restrict__ size) {
  const uint32_t id = lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= hi) return;
  const SahNode& nd = nodes[id];
  size[id] = nd.kind == SAH_INTERIOR ? 1u + size[nd.child] + size[nd.child + 1] : nd.kind == SAH_LEAF ? 1u : sub_cnt[nd.child];
}

// preorder: the first child at i + 1, the second after the first child's subtree (:179-181)
__global__ void __launch_bounds__(256) sah_preorder_kernel(uint32_t lo, uint32_t hi, const SahNode* __restrict__ nodes, const uint32_t* __restrict__ size,
                                                           uint32_t* __restrict__ pre) {
  const uint32_t id = lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= hi) return;
  const SahNode& nd = nodes[id];
  if (nd.kind != SAH_INTERIOR) return;
  pre[nd.child] = pre[id] + 1u;
  pre[nd.child + 1] = pre[id] + 1u + size[nd.child];
}

// one warp per BFS node: its record, or the records of its subtree moved into place
__global__ void __launch_bounds__(256) sah_emit_kernel(uint32_t n_bfs, const SahNode* __restrict__ nodes, const uint32_t* __restrict__ pre,
                                                       const uint32_t* __restrict__ sub_cnt, const float4* __restrict__ scratch, float4* __restrict__ out) {
  const uint32_t id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (id >= n_bfs) return;
  const SahNode& nd = nodes[id];
  const uint32_t at = pre[id];
  if (nd.kind == SAH_SUBTREE) {
    const float4* src = scratch + 4 * (size_t)nd.start;
    for (uint32_t r = lane; r < sub_cnt[nd.child]; r += 32) {
      float4 b = src[2 * r + 1];
      if ((__float_as_uint(b.w) & 0xffffu) == 0) b.z = __uint_as_float(__float_as_uint(b.z) + at);
      out[2 * (size_t)(at + r)] = src[2 * r];
      out[2 * (size_t)(at + r) + 1] = b;
    }
  } else if (lane == 0) {
    if (nd.kind == SAH_INTERIOR) put_record(out + 2 * (size_t)at, nd.box, pre[nd.child + 1], 0, nd.dim);
    else put_record(out + 2 * (size_t)at, nd.box, nd.start, nd.end - nd.start, 0);  // :86-94
  }
}

__global__ void __launch_bounds__(256) sah_perm_kernel(uint32_t n, const Prim* __restrict__ P, uint32_t* __restrict__ perm) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) perm[i] = P[i].id;
}

}  // namespace

// Builds ptrs_host::build_bvh(bounds, max_prims, 1) over n primitives given as device arrays in the caller's order.  On
// success *nodes_out holds *n_nodes_out 32-byte records in the reference's depth-first preorder (as float4 pairs),
// *perm_out the primitive order (BVH position -> caller index), and *max_depth_out the builder's max_depth (the root
// is 1).  A tree found to have nodes deeper than depth_limit is not finished: *max_depth_out is then larger than
// depth_limit and the outputs are empty.  Outputs are stream-ordered allocations the caller frees with cudaFreeAsync.
// Returns a cudaError_t.
int build_sah_bvh_on_device(cudaStream_t st, uint32_t n, const uint32_t* d_prim_vertex, const float* d_pos, int max_prims, uint32_t depth_limit,
                            float4** nodes_out, uint32_t* n_nodes_out, uint32_t** perm_out, uint32_t* max_depth_out) {
  *nodes_out = nullptr;
  *perm_out = nullptr;
  *n_nodes_out = 0;
  *max_depth_out = 0;
  if (n == 0) return cudaSuccess;
  const bool debug = std::getenv("PTRS_BVH_DEBUG") != nullptr;  // phase trace on stderr (synchronises between phases)
  auto t_phase = std::chrono::steady_clock::now();
  auto phase = [&](const char* what) {
    if (!debug) return;
    cudaStreamSynchronize(st);
    const auto t_now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "sah build: %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t_now - t_phase).count());
    t_phase = t_now;
  };
  cudaError_t e = cudaSuccess;
  auto ok = [&](cudaError_t r) {
    if (e == cudaSuccess && r != cudaSuccess) e = r;
    return e == cudaSuccess;
  };
  std::vector<void*> owned;  // working memory, released at the end
  auto take = [&](auto** p, size_t count) {
    *p = nullptr;
    if (ok(pool_alloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(**p), st))) owned.push_back(*p);
  };
  const uint32_t max_active = n / (SAH_SMALL + 1) + 1;  // nodes of one level are disjoint and larger than SAH_SMALL
  Prim* P = nullptr;
  uint32_t *seg = nullptr, *seg_next = nullptr, *flag = nullptr, *scan = nullptr, *right = nullptr, *active = nullptr, *next_active = nullptr;
  uint32_t *sub_list = nullptr, *sub_cnt = nullptr;
  SegAcc* acc = nullptr;
  SegPlan* plan = nullptr;
  Counters* ctr = nullptr;
  float4* scratch = nullptr;
  take(&P, n);
  take(&seg, n);
  take(&seg_next, n);
  take(&flag, n);
  take(&scan, n);
  take(&right, n);
  take(&active, max_active);
  take(&next_active, max_active);
  take(&sub_list, n);
  take(&sub_cnt, n);
  take(&acc, max_active);
  take(&plan, max_active);
  take(&ctr, 1);
  take(&scratch, 4 * (size_t)n);
  size_t scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, flag, scan, (int)n, st);
  char* scan_tmp = nullptr;
  take(&scan_tmp, scan_bytes);
  // BFS nodes: grown as levels need them (a level of k nodes adds at most 2k)
  uint32_t cap = 4 * max_active + 64;
  SahNode* nodes = nullptr;
  ok(pool_alloc(reinterpret_cast<void**>(&nodes), (size_t)cap * sizeof(SahNode), st));
  const int grid = 148 * 8;
  const int tiles = (int)std::min<uint32_t>(grid, (n + SAH_TILE - 1) / SAH_TILE);
  Counters h{1u, 0u, 0u, 1u};
  std::vector<uint32_t> lvl{0u, 1u};  // BFS ids of level L: [lvl[L], lvl[L + 1])
  phase("allocation");
  if (e == cudaSuccess) {
    sah_prims_kernel<<<grid, 256, 0, st>>>(n, d_prim_vertex, d_pos, P);
    SahNode root{};
    root.start = 0;
    root.end = n;
    root.depth = 1;
    uint32_t n_active = 0;
    if (n > SAH_SMALL) {
      root.kind = SAH_PENDING;
      n_active = 1;
      const uint32_t zero = 0;
      ok(cudaMemcpyAsync(active, &zero, 4, cudaMemcpyHostToDevice, st));
      ok(cudaMemsetAsync(seg, 0, (size_t)n * 4, st));
    } else {
      root.kind = SAH_SUBTREE;
      root.child = 0;
      h.n_sub = 1;
      const uint32_t zero = 0;
      ok(cudaMemcpyAsync(sub_list, &zero, 4, cudaMemcpyHostToDevice, st));
    }
    ok(cudaMemcpyAsync(nodes, &root, sizeof(root), cudaMemcpyHostToDevice, st));
    ok(cudaMemcpyAsync(ctr, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    uint32_t level = 0;
    while (e == cudaSuccess && n_active > 0) {
      if (h.n_bfs + 2 * n_active > cap) {
        const uint32_t want = std::max(2 * cap, h.n_bfs + 2 * n_active);
        SahNode* grown = nullptr;
        if (ok(pool_alloc(reinterpret_cast<void**>(&grown), (size_t)want * sizeof(SahNode), st))) {
          ok(cudaMemcpyAsync(grown, nodes, (size_t)h.n_bfs * sizeof(SahNode), cudaMemcpyDeviceToDevice, st));
          cudaFreeAsync(nodes, st);
          nodes = grown;
          cap = want;
        }
      }
      h.n_next = 0;
      ok(cudaMemcpyAsync(ctr, &h, sizeof(h), cudaMemcpyHostToDevice, st));
      const int ga = (int)((n_active + 127) / 128);
      sah_acc_init_kernel<<<ga, 128, 0, st>>>(n_active, acc);
      sah_box_kernel<<<tiles, 256, 0, st>>>(n, P, seg, acc);
      sah_decide_kernel<<<ga, 128, 0, st>>>(n_active, active, nodes, P, acc, plan, ctr, next_active, sub_list);
      sah_bucket_kernel<<<tiles, 256, 0, st>>>(n, P, seg, plan, acc);
      sah_cost_kernel<<<ga, 128, 0, st>>>(n_active, nodes, acc, plan, max_prims, ctr, next_active, sub_list);
      sah_flag_kernel<<<grid, 256, 0, st>>>(n, P, seg, plan, flag);
      ok(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, flag, scan, (int)n, st));
      sah_pair_kernel<<<grid, 256, 0, st>>>(n, seg, plan, nodes, flag, scan, right);
      sah_swap_kernel<<<grid, 256, 0, st>>>(n, P, seg, plan, nodes, flag, scan, right, seg_next);
      ok(cudaMemcpyAsync(&h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
      ok(cudaStreamSynchronize(st));
      ok(cudaGetLastError());
      std::swap(seg, seg_next);
      std::swap(active, next_active);
      n_active = h.n_next;
      lvl.push_back(h.n_bfs);
      ++level;
      if (n_active > 0 && level + 1 > depth_limit) {  // the next level's nodes are too deep: stop here
        *max_depth_out = level + 1;
        break;
      }
    }
    phase("levels");
  }
  const bool finished = e == cudaSuccess && *max_depth_out == 0;
  uint32_t n_records = 0;
  float4* out = nullptr;
  uint32_t* perm = nullptr;
  if (finished) {
    if (h.n_sub > 0) sah_small_kernel<<<(h.n_sub + 127) / 128, 128, 0, st>>>(h.n_sub, sub_list, nodes, P, max_prims, scratch, sub_cnt, ctr);
    phase("subtrees");
    uint32_t *size = nullptr, *pre = nullptr;
    take(&size, h.n_bfs);
    take(&pre, h.n_bfs);
    if (e == cudaSuccess) {
      for (size_t L = lvl.size() - 1; L-- > 0;) {
        const uint32_t lo = lvl[L], hi = lvl[L + 1];
        if (hi > lo) sah_size_kernel<<<(hi - lo + 255) / 256, 256, 0, st>>>(lo, hi, nodes, sub_cnt, size);
      }
      ok(cudaMemsetAsync(pre, 0, 4, st));
      for (size_t L = 0; L + 1 < lvl.size(); ++L) {
        const uint32_t lo = lvl[L], hi = lvl[L + 1];
        if (hi > lo) sah_preorder_kernel<<<(hi - lo + 255) / 256, 256, 0, st>>>(lo, hi, nodes, size, pre);
      }
      ok(cudaMemcpyAsync(&n_records, size, 4, cudaMemcpyDeviceToHost, st));
      ok(cudaMemcpyAsync(&h.max_depth, &ctr->max_depth, 4, cudaMemcpyDeviceToHost, st));
      ok(cudaStreamSynchronize(st));
    }
    if (e == cudaSuccess) ok(pool_alloc(reinterpret_cast<void**>(&out), (size_t)n_records * 32, st));
    if (e == cudaSuccess) ok(pool_alloc(reinterpret_cast<void**>(&perm), (size_t)n * 4, st));
    if (e == cudaSuccess) {
      sah_emit_kernel<<<(h.n_bfs + 7) / 8, 256, 0, st>>>(h.n_bfs, nodes, pre, sub_cnt, scratch, out);
      sah_perm_kernel<<<grid, 256, 0, st>>>(n, P, perm);
      ok(cudaGetLastError());
    }
    phase("preorder, emission");
  }
  for (void* p : owned) cudaFreeAsync(p, st);
  if (nodes) cudaFreeAsync(nodes, st);
  if (e != cudaSuccess || !finished) {
    if (out) cudaFreeAsync(out, st);
    if (perm) cudaFreeAsync(perm, st);
    return (int)e;
  }
  *nodes_out = out;
  *perm_out = perm;
  *n_nodes_out = n_records;
  *max_depth_out = h.max_depth;
  return (int)cudaSuccess;
}

}  // namespace ptrs
