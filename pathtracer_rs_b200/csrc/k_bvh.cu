// BVH construction on the device (SURVEY.md §8f-1): replaces the host's recursive SAH build
// (src/pathtracer/accelerator.rs:103-346) when the caller hands over unordered primitives.
//
// 63-bit Morton codes of the primitive centroids -> radix sort -> tree topology -> subtrees of at most 4 primitives
// collapse into leaves where the reference builder's own cost criterion says so (max_prims_in_node = 4) -> emission
// into the traversal layout of dev_accel.cuh: 32-byte LinearBVHNode records, the two children of an interior node side
// by side (64-byte pairs), pairs numbered depth-first so a subtree is contiguous in memory.  `axis` is the axis along
// which the two children's box centres differ most and the first child is the lower one, which is what the
// traversal's near-child rule dir_is_neg[axis] (accelerator.rs:393-404) assumes.
//
// Two topologies over the same sorted sequence:
//   PLOC (default)   bottom-up clustering by smallest merged surface area within a window of the Morton order
//                    (Meister & Bittner 2018): SAH-quality trees — measured against the reference-built SAH tree:
//                    4K atrium 5 - 15 % FASTER to traverse, 1 M-triangle field equal, 10 M-triangle terrain 14 % slower
//   radix tree       Karras 2012, one thread per internal node + bottom-up boxes with one atomic per node
//                    (PTRS_BVH_BUILDER=lbvh): a third of the build time, 10 - 30 % slower to traverse than PLOC
//
// Every kernel is a streaming pass over HBM-resident arrays (24-68 B per primitive); the sort is
// cub::DeviceRadixSort (library code, like cuBLAS for a plain GEMM).  The tree differs from the reference's SAH
// tree, so visit counts differ, but closest hits do not: the triangle test is the same code on the same vertices.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "launch.hpp"
#include "wavefront.cuh"

namespace ptrs {

namespace {

// order-preserving float <-> uint map for atomicMin / atomicMax on floats
__device__ __forceinline__ uint32_t f2o(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float o2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

// One 32-byte record (= one DRAM sector) per radix-tree node, so that a refit step touches three sectors (the
// parent's record, the sibling's box, the parent's box) instead of a dozen scattered 4-byte fields.
struct __align__(32) TreeNode {  // internal nodes [0, n-1); leaves are addressed as (n - 1 + sorted position)
  uint32_t left, right, parent;
  uint32_t first, last;   // sorted range covered
  uint32_t arrivals;      // refit: children finished so far
  uint32_t n_interior;    // emitted interior nodes in the subtree (0 when the subtree collapses into a leaf)
  uint32_t left_count;    // PLOC: primitives below `left` (what a primitive of the right subtree adds to its depth-first position)
};
struct __align__(32) NodeBox {
  float4 mn, mx;  // xyz used
};
struct BuildArrays {
  float4* pb_min;  // per primitive, caller order: bounds min / max
  float4* pb_max;
  uint64_t* keys;  // per primitive, sorted order
  uint32_t* perm;  // sorted position -> caller's primitive index
  TreeNode* node;         // n - 1
  uint32_t* leaf_parent;  // n
  NodeBox* box;           // 2n - 1
  uint32_t* cbounds;      // 6 ordered uints: centroid bounds
  uint32_t* leaf_pos;     // PLOC: sorted position -> depth-first position of the primitive (null: the two coincide)
};

__global__ void __launch_bounds__(256) prim_bounds_kernel(const uint32_t* __restrict__ prim_vertex, const float* __restrict__ pos, uint32_t n, BuildArrays A) {
  float cmin[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, cmax[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float mn[3], mx[3];
    for (int k = 0; k < 3; ++k) {
      const uint32_t v = prim_vertex[3 * (size_t)i + k];
      for (int a = 0; a < 3; ++a) {
        const float x = __ldg(pos + 3 * (size_t)v + a);
        mn[a] = k == 0 ? x : fminf(mn[a], x);
        mx[a] = k == 0 ? x : fmaxf(mx[a], x);
      }
    }
    A.pb_min[i] = make_float4(mn[0], mn[1], mn[2], 0.f);
    A.pb_max[i] = make_float4(mx[0], mx[1], mx[2], 0.f);
    for (int a = 0; a < 3; ++a) {
      const float c = 0.5f * mn[a] + 0.5f * mx[a];
      cmin[a] = fminf(cmin[a], c);
      cmax[a] = fmaxf(cmax[a], c);
    }
  }
  for (int a = 0; a < 3; ++a) {
    for (int o = 16; o > 0; o >>= 1) {
      cmin[a] = fminf(cmin[a], __shfl_xor_sync(0xffffffffu, cmin[a], o));
      cmax[a] = fmaxf(cmax[a], __shfl_xor_sync(0xffffffffu, cmax[a], o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&A.cbounds[a], f2o(cmin[a]));
      atomicMax(&A.cbounds[3 + a], f2o(cmax[a]));
    }
  }
}

__device__ __forceinline__ uint64_t spread21(uint64_t x) {  // 21 bits -> every third bit
  x &= 0x1fffffull;
  x = (x | (x << 32)) & 0x1f00000000ffffull;
  x = (x | (x << 16)) & 0x1f0000ff0000ffull;
  x = (x | (x << 8)) & 0x100f00f00f00f00full;
  x = (x | (x << 4)) & 0x10c30c30c30c30c3ull;
  x = (x | (x << 2)) & 0x1249249249249249ull;
  return x;
}

__global__ void __launch_bounds__(256) morton_kernel(uint32_t n, BuildArrays A) {
  float lo[3], inv[3];
  for (int a = 0; a < 3; ++a) {
    lo[a] = o2f(A.cbounds[a]);
    const float ext = o2f(A.cbounds[3 + a]) - lo[a];
    inv[a] = ext > 0.f ? 2097152.0f / ext : 0.f;  // 2^21 cells per axis
  }
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 mn = A.pb_min[i], mx = A.pb_max[i];
    const float c[3] = {0.5f * mn.x + 0.5f * mx.x, 0.5f * mn.y + 0.5f * mx.y, 0.5f * mn.z + 0.5f * mx.z};
    uint64_t q[3];
    for (int a = 0; a < 3; ++a) q[a] = (uint64_t)fminf(fmaxf((c[a] - lo[a]) * inv[a], 0.f), 2097151.0f);
    A.keys[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    A.perm[i] = i;
  }
}

// common-prefix length of sorted keys i and j, ties broken by position (Karras 2012, section 4)
__device__ __forceinline__ int prefix_len(const uint64_t* __restrict__ keys, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  const uint64_t a = keys[i], b = keys[j];
  return a == b ? 64 + __clz((uint32_t)i ^ (uint32_t)j) : __clzll((long long)(a ^ b));
}

__global__ void __launch_bounds__(256) radix_tree_kernel(const uint64_t* __restrict__ keys, int n, BuildArrays A) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n - 1; i += gridDim.x * blockDim.x) {
    const int d = prefix_len(keys, n, i, i + 1) - prefix_len(keys, n, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = prefix_len(keys, n, i, i - d);
    int lmax = 2;
    while (prefix_len(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
      if (prefix_len(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = prefix_len(keys, n, i, j);
    int s = 0, t = l;
    do {
      t = (t + 1) >> 1;
      if (prefix_len(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const uint32_t lc = lo == gamma ? (uint32_t)(n - 1 + gamma) : (uint32_t)gamma;
    const uint32_t rc = hi == gamma + 1 ? (uint32_t)(n - 1 + gamma + 1) : (uint32_t)(gamma + 1);
    TreeNode& nd = A.node[i];
    nd.left = lc;
    nd.right = rc;
    nd.first = (uint32_t)lo;
    nd.last = (uint32_t)hi;
    nd.arrivals = 0u;
    nd.n_interior = 0u;
    if (lc >= (uint32_t)(n - 1)) A.leaf_parent[lc - (uint32_t)(n - 1)] = (uint32_t)i;
    else A.node[lc].parent = (uint32_t)i;
    if (rc >= (uint32_t)(n - 1)) A.leaf_parent[rc - (uint32_t)(n - 1)] = (uint32_t)i;
    else A.node[rc].parent = (uint32_t)i;
    if (i == 0) nd.parent = 0xffffffffu;
  }
}

#define PT_BVH_MAX_LEAF 4u  // BVH::new(.., &4), importer/mitsuba.rs:362

__device__ __forceinline__ float box_area(float4 mn, float4 mx) {
  const float dx = mx.x - mn.x, dy = mx.y - mn.y, dz = mx.z - mn.z;
  return 2.0f * (dx * dy + dy * dz + dz * dx);
}

// Bottom-up pass over the radix tree: boxes, and which subtrees become leaves.  A subtree of at most PT_BVH_MAX_LEAF
// primitives whose two halves are leaves themselves collapses into ONE leaf only if that is not more expensive than
// keeping the split, by the reference builder's own criterion (accelerator.rs:240-254: leaf iff
// 1 + (n0 A0 + n1 A1) / A >= n): a Morton split that separates two clusters of triangles stays a node instead of
// becoming a 4-triangle leaf whose box is mostly empty.
__global__ void __launch_bounds__(256) refit_kernel(uint32_t n, BuildArrays A) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const uint32_t prim = A.perm[j];
    uint32_t node = n - 1 + j;
    float4 mn = A.pb_min[prim], mx = A.pb_max[prim];
    A.box[node] = NodeBox{mn, mx};
    if (n == 1) return;
    uint32_t p = A.leaf_parent[j];
    uint32_t ni_self = 0;   // emitted interior nodes below (and including) `node`
    uint32_t cnt_self = 1;  // primitives below `node`
    for (;;) {
      __threadfence();
      TreeNode* pn = A.node + p;
      if (atomicAdd(&pn->arrivals, 1u) == 0u) break;  // the sibling subtree is not finished: its thread continues
      __threadfence();
      const uint4 w0 = __ldcg(reinterpret_cast<const uint4*>(pn));      // left, right, parent, first
      const uint4 w1 = __ldcg(reinterpret_cast<const uint4*>(pn) + 1);  // last, arrivals, n_interior, pad
      const uint32_t other = w0.x == node ? w0.y : w0.x;
      const float4 omn = __ldcg(&A.box[other].mn), omx = __ldcg(&A.box[other].mx);
      const float a_self = box_area(mn, mx), a_other = box_area(omn, omx);
      mn = make_float4(fminf(mn.x, omn.x), fminf(mn.y, omn.y), fminf(mn.z, omn.z), 0.f);
      mx = make_float4(fmaxf(mx.x, omx.x), fmaxf(mx.y, omx.y), fmaxf(mx.z, omx.z), 0.f);
      A.box[p] = NodeBox{mn, mx};
      const uint32_t count = w1.x - w0.w + 1u;
      const uint32_t ni_other = other < n - 1 ? __ldcg(&A.node[other].n_interior) : 0u;
      bool leaf = count <= PT_BVH_MAX_LEAF && ni_self == 0u && ni_other == 0u;
      if (leaf) {
        const float a = box_area(mn, mx);
        const float cost = 1.0f + ((float)cnt_self * a_self + (float)(count - cnt_self) * a_other) / a;
        leaf = !(cost < (float)count);  // also a leaf when the box has no area (cost is NaN or inf)
      }
      const uint32_t ni = leaf ? 0u : 1u + ni_self + ni_other;
      pn->n_interior = ni;
      ni_self = ni;
      cnt_self = count;
      node = p;
      p = w0.z;
      if (p == 0xffffffffu) break;
    }
  }
}


// ---- PLOC: parallel locally-ordered clustering (Meister & Bittner 2018) ---------------------------------------------
// The radix tree above splits at Morton-code bit boundaries, i.e. at spatial medians of alternating axes whatever the
// geometry looks like; the reference's builder chooses every split by the surface-area heuristic (accelerator.rs:
// 156-307).  PLOC gets SAH-quality trees out of the same sorted sequence, bottom-up: every cluster looks PLOC_R places
// to either side of its position in the (Morton-ordered) cluster sequence for the neighbour whose union with it has the
// smallest surface area; two clusters that chose each other merge into a new node that takes the lower one's place; the
// sequence is compacted; repeat until one cluster is left (about 35 rounds for 10^7 primitives).  Counts, the leaf
// decision (same criterion as refit_kernel) and the interior-node counts are known at merge time, so there is no
// separate refit pass.  Merged clusters are not contiguous ranges of the sorted order, so the primitives' final order
// is the depth-first order of the finished tree (ploc_positions_kernel).
#define PLOC_R 16
#define PLOC_BLOCK 256
#define PLOC_NONE 0xffffffffu
#define PLOC_MAX_ROUNDS 512

__global__ void __launch_bounds__(256) ploc_init_kernel(uint32_t n, BuildArrays A, uint32_t* __restrict__ cid) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const uint32_t prim = A.perm[j];
    A.box[n - 1 + j] = NodeBox{A.pb_min[prim], A.pb_max[prim]};
    cid[j] = n - 1 + j;
  }
}

// nearest neighbour of every cluster within PLOC_R positions; the candidates' boxes are staged once per block in shared
// memory.  Distance = area of the union (symmetric bit for bit: min / max commute).  Ties — the rule on regular meshes,
// where many unions have the same area — are broken by a key that both ends of a pair compute alike: the nearer position
// first, then the pair whose lower position is even, then the lower position.  The pair with the smallest (distance, key)
// overall therefore always chooses each other (every round merges), and a run of equal distances pairs up as (0,1), (2,3),
// ... and halves per round instead of peeling one pair off its end.
__global__ void __launch_bounds__(PLOC_BLOCK) ploc_nn_kernel(uint32_t m, const uint32_t* __restrict__ cid, const NodeBox* __restrict__ box, uint32_t* __restrict__ nn) {
  __shared__ float4 s_mn[PLOC_BLOCK + 2 * PLOC_R], s_mx[PLOC_BLOCK + 2 * PLOC_R];
  for (uint32_t base = blockIdx.x * PLOC_BLOCK; base < m; base += gridDim.x * PLOC_BLOCK) {
    for (uint32_t t = threadIdx.x; t < PLOC_BLOCK + 2 * PLOC_R; t += PLOC_BLOCK) {
      const long long g = (long long)base - PLOC_R + (long long)t;
      if (g >= 0 && g < (long long)m) {
        const uint32_t id = cid[g];
        s_mn[t] = box[id].mn;
        s_mx[t] = box[id].mx;
      }
    }
    __syncthreads();
    const uint32_t i = base + threadIdx.x;
    if (i < m) {
      const int me = (int)threadIdx.x + PLOC_R;
      const float4 mn = s_mn[me], mx = s_mx[me];
      float best = CUDART_INF_F;
      uint32_t best_j = PLOC_NONE;
      auto consider = [&](int d) {  // candidates arrive in tie-break order, so a strict comparison keeps the preferred one
        const long long j = (long long)i + d;
        if (j < 0 || j >= (long long)m) return;
        const float4 omn = s_mn[me + d], omx = s_mx[me + d];
        const float4 umn = make_float4(fminf(mn.x, omn.x), fminf(mn.y, omn.y), fminf(mn.z, omn.z), 0.f);
        const float4 umx = make_float4(fmaxf(mx.x, omx.x), fmaxf(mx.y, omx.y), fmaxf(mx.z, omx.z), 0.f);
        const float a = fminf(box_area(umn, umx), 3.0e38f);  // NaN / inf areas (degenerate input) still order
        if (a < best) {
          best = a;
          best_j = (uint32_t)j;
        }
      };
#pragma unroll 4
      for (int d = 1; d <= PLOC_R; ++d) {
        // pair (i - d, i) has lower position i - d, pair (i, i + d) has lower position i: even lower position first, and
        // when both have the same parity (d even) the lower one
        const bool up_first = (d & 1) && !(i & 1u);
        consider(up_first ? d : -d);
        consider(up_first ? -d : d);
      }
      nn[i] = best_j;
    }
    __syncthreads();
  }
}

// mutual pairs merge: the lower position creates the node (ids are handed out downwards from n - 2, so the last merge,
// the root, is node 0 as in the radix tree) and keeps its place, the upper position drops out of the sequence
__global__ void __launch_bounds__(256) ploc_merge_kernel(uint32_t m, uint32_t n, const uint32_t* __restrict__ cid, const uint32_t* __restrict__ nn, BuildArrays A,
                                                         uint32_t* __restrict__ counter, uint32_t* __restrict__ cid_out, uint32_t* __restrict__ keep) {
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t base = blockIdx.x * blockDim.x; base < m; base += gridDim.x * blockDim.x) {  // warp-uniform trip count
    const uint32_t i = base + threadIdx.x;
    uint32_t j = PLOC_NONE;
    bool creates = false;
    if (i < m) {
      j = nn[i];
      const bool mutual = j != PLOC_NONE && nn[j] == i;
      if (!mutual) {
        cid_out[i] = cid[i];
        keep[i] = 1u;
      } else if (i > j) {
        keep[i] = 0u;
      } else {
        creates = true;
      }
    }
    // node ids: one atomicAdd per warp
    const uint32_t cmask = __ballot_sync(0xffffffffu, creates);
    uint32_t id0 = 0;
    if (cmask != 0u && lane == (uint32_t)(__ffs(cmask) - 1)) id0 = atomicAdd(counter, (uint32_t)__popc(cmask));
    id0 = __shfl_sync(0xffffffffu, id0, cmask ? __ffs(cmask) - 1 : 0);
    if (!creates) continue;
    const uint32_t l = cid[i], r = cid[j];
    const uint32_t id = n - 2u - (id0 + (uint32_t)__popc(cmask & ((1u << lane) - 1u)));
    const float4 lmn = A.box[l].mn, lmx = A.box[l].mx, rmn = A.box[r].mn, rmx = A.box[r].mx;
    const float4 mn = make_float4(fminf(lmn.x, rmn.x), fminf(lmn.y, rmn.y), fminf(lmn.z, rmn.z), 0.f);
    const float4 mx = make_float4(fmaxf(lmx.x, rmx.x), fmaxf(lmx.y, rmx.y), fmaxf(lmx.z, rmx.z), 0.f);
    uint32_t cl = 1u, cr = 1u, nil = 0u, nir = 0u;
    if (l < n - 1) {  // TreeNode::last holds the primitive COUNT until ploc_positions_kernel turns it into a range
      cl = A.node[l].last;
      nil = A.node[l].n_interior;
      A.node[l].parent = id;
    } else {
      A.leaf_parent[l - (n - 1)] = id;
    }
    if (r < n - 1) {
      cr = A.node[r].last;
      nir = A.node[r].n_interior;
      A.node[r].parent = id;
    } else {
      A.leaf_parent[r - (n - 1)] = id;
    }
    const uint32_t count = cl + cr;
    bool leaf = count <= PT_BVH_MAX_LEAF && nil == 0u && nir == 0u;
    if (leaf) {  // accelerator.rs:240-254, as in refit_kernel
      const float cost = 1.0f + ((float)cl * box_area(lmn, lmx) + (float)cr * box_area(rmn, rmx)) / box_area(mn, mx);
      leaf = !(cost < (float)count);
    }
    TreeNode nd;
    nd.left = l;
    nd.right = r;
    nd.parent = 0xffffffffu;
    nd.first = 0u;
    nd.last = count;
    nd.arrivals = 0u;
    nd.n_interior = leaf ? 0u : 1u + nil + nir;
    nd.left_count = cl;
    A.node[id] = nd;
    A.box[id] = NodeBox{mn, mx};
    cid_out[i] = id;
    keep[i] = 1u;
  }
}

__global__ void __launch_bounds__(256) ploc_compact_kernel(uint32_t m, const uint32_t* __restrict__ cid_out, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ rank,
                                                           uint32_t* __restrict__ cid_next, uint32_t* __restrict__ m_next) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    if (keep[i]) cid_next[rank[i]] = cid_out[i];
    if (i == m - 1) *m_next = rank[i] + keep[i];
  }
}

// depth-first position of every node's first primitive: on the way up to the root, a node that hangs in a right subtree
// comes after everything below the left sibling.  Interior nodes get their primitive range (first, last) as the radix
// tree has it by construction; leaves get their final position and the primitive order follows.
__global__ void __launch_bounds__(256) ploc_positions_kernel(uint32_t n, BuildArrays A, const uint32_t* __restrict__ perm_sorted, uint32_t* __restrict__ perm_final) {
  for (uint32_t x = blockIdx.x * blockDim.x + threadIdx.x; x < 2u * n - 1u; x += gridDim.x * blockDim.x) {
    uint32_t c = x, first = 0u;
    uint32_t p = x < n - 1 ? A.node[x].parent : A.leaf_parent[x - (n - 1)];
    while (p != 0xffffffffu) {
      const uint4 w0 = *reinterpret_cast<const uint4*>(A.node + p);  // left, right, parent, first
      if (w0.y == c) first += A.node[p].left_count;
      c = p;
      p = w0.z;
    }
    if (x < n - 1) {
      const uint32_t count = A.node[x].last;
      A.node[x].first = first;
      A.node[x].last = first + count - 1u;
    } else {
      A.leaf_pos[x - (n - 1)] = first;
      perm_final[first] = perm_sorted[x - (n - 1)];
    }
  }
}

struct NodeRec {  // the reference's LinearBVHNode (accelerator.rs:83-95) as two float4
  float4 a, b;
};
__device__ __forceinline__ NodeRec make_node(float4 mn, float4 mx, uint32_t offset, uint32_t n_prims, uint32_t axis) {
  NodeRec r;
  r.a = make_float4(mn.x, mn.y, mn.z, mx.x);
  r.b = make_float4(mx.y, mx.z, __uint_as_float(offset), __uint_as_float((n_prims & 0xffffu) | (axis << 16)));
  return r;
}

// one thread per emitted interior node: depth-first pair number from the path to the root, then the two child records
// *max_depth receives the largest (number of interior ancestors + 1) over the emitted interior nodes: the most pending
// stack entries a traversal of this tree can hold
__global__ void __launch_bounds__(256) emit_kernel(uint32_t n, BuildArrays A, float4* __restrict__ nodes, uint32_t* __restrict__ max_depth) {
  uint32_t deepest = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n - 1; i += gridDim.x * blockDim.x) {
    const TreeNode self = A.node[i];
    if (self.n_interior == 0) continue;
    uint32_t pair = 1, depth = 1;
    for (uint32_t c = i, p = self.parent; c != 0;) {
      const TreeNode pn = A.node[p];
      pair += 1;
      depth += 1;
      if (pn.right == c && pn.left < n - 1) pair += A.node[pn.left].n_interior;
      c = p;
      p = pn.parent;
    }
    deepest = max(deepest, depth);
    const uint32_t l = self.left, r = self.right;
    const uint32_t l_int = l < n - 1 ? A.node[l].n_interior : 0u, r_int = r < n - 1 ? A.node[r].n_interior : 0u;
    const float4 lmn = A.box[l].mn, lmx = A.box[l].mx, rmn = A.box[r].mn, rmx = A.box[r].mx;
    // split axis: where the children's box centres differ most; the lower child goes first
    const float dc[3] = {(rmn.x + rmx.x) - (lmn.x + lmx.x), (rmn.y + rmx.y) - (lmn.y + lmx.y), (rmn.z + rmx.z) - (lmn.z + lmx.z)};
    uint32_t axis = 0;
    if (fabsf(dc[1]) > fabsf(dc[axis])) axis = 1;
    if (fabsf(dc[2]) > fabsf(dc[axis])) axis = 2;
    const bool swap = dc[axis] < 0.f;
    auto child = [&](uint32_t c, uint32_t c_int, uint32_t c_pair, float4 mn, float4 mx) {
      if (c_int) {
        const uint32_t gl = A.node[c].left, gr = A.node[c].right;
        const float4 gmn_l = A.box[gl].mn, gmx_l = A.box[gl].mx, gmn_r = A.box[gr].mn, gmx_r = A.box[gr].mx;
        const float g[3] = {(gmn_r.x + gmx_r.x) - (gmn_l.x + gmx_l.x), (gmn_r.y + gmx_r.y) - (gmn_l.y + gmx_l.y), (gmn_r.z + gmx_r.z) - (gmn_l.z + gmx_l.z)};
        uint32_t ax = 0;
        if (fabsf(g[1]) > fabsf(g[ax])) ax = 1;
        if (fabsf(g[2]) > fabsf(g[ax])) ax = 2;
        return make_node(mn, mx, 2u * c_pair, 0u, ax);
      }
      const uint32_t f = c < n - 1 ? A.node[c].first : (A.leaf_pos ? A.leaf_pos[c - (n - 1)] : c - (n - 1));
      const uint32_t cnt = c < n - 1 ? A.node[c].last - A.node[c].first + 1u : 1u;
      return make_node(mn, mx, f, cnt, 0u);
    };
    const NodeRec ln = child(l, l_int, pair + 1, lmn, lmx), rn = child(r, r_int, pair + 1 + l_int, rmn, rmx);
    const NodeRec first = swap ? rn : ln, second = swap ? ln : rn;
    nodes[4 * (size_t)pair] = first.a;
    nodes[4 * (size_t)pair + 1] = first.b;
    nodes[4 * (size_t)pair + 2] = second.a;
    nodes[4 * (size_t)pair + 3] = second.b;
    if (i == 0) {
      const NodeRec root = make_node(A.box[0].mn, A.box[0].mx, 2u, 0u, axis);
      nodes[0] = root.a;
      nodes[1] = root.b;
      nodes[2] = make_float4(0.f, 0.f, 0.f, 0.f);
      nodes[3] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  for (int o = 16; o > 0; o >>= 1) deepest = max(deepest, __shfl_xor_sync(0xffffffffu, deepest, o));
  if ((threadIdx.x & 31) == 0 && deepest) atomicMax(max_depth, deepest);
}

// scene of at most PT_BVH_MAX_LEAF primitives: the root is the only node, a leaf
__global__ void single_leaf_kernel(uint32_t n, BuildArrays A, float4* __restrict__ nodes) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float4 mn = A.pb_min[0], mx = A.pb_max[0];
  for (uint32_t i = 1; i < n; ++i) {
    const float4 a = A.pb_min[i], b = A.pb_max[i];
    mn = make_float4(fminf(mn.x, a.x), fminf(mn.y, a.y), fminf(mn.z, a.z), 0.f);
    mx = make_float4(fmaxf(mx.x, b.x), fmaxf(mx.y, b.y), fmaxf(mx.z, b.z), 0.f);
  }
  const NodeRec root = make_node(mn, mx, 0u, n, 0u);
  nodes[0] = root.a;
  nodes[1] = root.b;
  nodes[2] = nodes[3] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// triangles in BVH order: the same 3 x float4 (+ metadata in .w) and index records ptrs_scene_create lays out on the host
__global__ void __launch_bounds__(256) assemble_tris_kernel(uint32_t n, const uint32_t* __restrict__ perm, const uint32_t* __restrict__ prim_vertex,
                                                            const float* __restrict__ pos, const int32_t* __restrict__ prim_mesh,
                                                            const int32_t* __restrict__ prim_material, const int32_t* __restrict__ prim_area_light,
                                                            const PtrsMesh* __restrict__ meshes, float4* __restrict__ tri_verts, uint4* __restrict__ tri_index,
                                                            uint32_t* __restrict__ inv_perm) {
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const uint32_t i = perm ? perm[k] : k;  // null perm: the caller's order is the BVH order (reference-built tree)
    if (inv_perm) inv_perm[i] = k;
    const int32_t mesh = prim_mesh[i];
    const PtrsMesh m = meshes[mesh];
    uint32_t meta2 = m.flags & 0xffu;
    if (m.alpha_tex >= 0) meta2 |= PT_TRI_ALPHA_BIT | ((uint32_t)m.alpha_tex << 9);
    const int32_t w[3] = {prim_material[i], prim_area_light[i], (int32_t)meta2};
    uint32_t v[3];
    for (int c = 0; c < 3; ++c) {
      v[c] = prim_vertex[3 * (size_t)i + c];
      tri_verts[3 * (size_t)k + c] = make_float4(__ldg(pos + 3 * (size_t)v[c]), __ldg(pos + 3 * (size_t)v[c] + 1), __ldg(pos + 3 * (size_t)v[c] + 2), __int_as_float(w[c]));
    }
    tri_index[k] = make_uint4(v[0], v[1], v[2], (uint32_t)mesh);
  }
}

// index validation of the caller's primitive arrays, so that every later kernel can trust them
__global__ void __launch_bounds__(256) validate_prims_kernel(uint32_t n, const uint32_t* __restrict__ prim_vertex, const int32_t* __restrict__ prim_mesh,
                                                             const int32_t* __restrict__ prim_material, const int32_t* __restrict__ prim_area_light,
                                                             uint32_t n_verts, uint32_t n_meshes, uint32_t n_materials, uint32_t n_lights,
                                                             const PtrsLight* __restrict__ lights, uint32_t* __restrict__ err) {
  uint32_t e = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (prim_mesh[i] < 0 || (uint32_t)prim_mesh[i] >= n_meshes || prim_material[i] < 0 || (uint32_t)prim_material[i] >= n_materials ||
        prim_area_light[i] >= (int32_t)n_lights)
      e |= 1u;
    else if (prim_area_light[i] >= 0 && lights[prim_area_light[i]].type != PTRS_LIGHT_AREA)  // area_le reads the light's ke texture
      e |= 4u;
    for (int k = 0; k < 3; ++k)
      if (prim_vertex[3 * (size_t)i + k] >= n_verts) e |= 2u;
  }
  if (e) atomicOr(err, e);
}

// ---- pair layout of a reference-built tree -------------------------------------------------------------------------
// The reference's flattened tree (accelerator.rs:348-357) is in depth-first preorder: first child at i + 1, second at
// `offset`.  The traversal layout places the children of the r-th interior node (in that same order) side by side in
// slots 2 (r + 1), 2 (r + 1) + 1, so the position of every record follows from an exclusive prefix count of interior
// nodes: one scan and one scatter pass instead of a serial walk on the host.
__global__ void __launch_bounds__(256) interior_flag_kernel(const float4* __restrict__ raw, uint32_t n, uint32_t* __restrict__ flag) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    flag[i] = (__float_as_uint(raw[2 * (size_t)i + 1].w) & 0xffffu) == 0 ? 1u : 0u;
}
__global__ void __launch_bounds__(256) pair_layout_kernel(const float4* __restrict__ raw, uint32_t n, const uint32_t* __restrict__ rank, float4* __restrict__ out) {
  auto place = [&](uint32_t j, uint32_t slot) {
    const float4 a = raw[2 * (size_t)j];
    float4 b = raw[2 * (size_t)j + 1];
    // n_prims (16 bits) and axis (0..2) only: LinearBVHNode's fourth byte is padding whose content is the caller's, and the
    // traversal tells "no node" from a node by bit 31 of this word (PT_NO_NODE, dev_accel.cuh)
    b.w = __uint_as_float(__float_as_uint(b.w) & 0x0003ffffu);
    if ((__float_as_uint(b.w) & 0xffffu) == 0) b.z = __uint_as_float(2u * (rank[j] + 1u));  // interior: where ITS children sit
    out[2 * (size_t)slot] = a;
    out[2 * (size_t)slot + 1] = b;
  };
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (i == 0) {
      place(0, 0);
      out[2] = make_float4(0.f, 0.f, 0.f, 0.f);
      out[3] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float4 b = raw[2 * (size_t)i + 1];
    if ((__float_as_uint(b.w) & 0xffffu) != 0) continue;
    const uint32_t k = 2u * (rank[i] + 1u);
    place(i + 1, k);
    place(__float_as_uint(b.z), k + 1);
  }
}

__global__ void remap_light_prims_kernel(PtrsLight* lights, uint32_t n_lights, const uint32_t* __restrict__ inv_perm) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_lights && lights[i].type == PTRS_LIGHT_AREA) lights[i].prim = (int32_t)inv_perm[lights[i].prim];
}

struct Arena {  // one stream-ordered allocation carved into 256-byte aligned arrays
  char* base = nullptr;
  size_t used = 0;
  template <class T>
  void take(T** p, size_t count) {
    if (base) *p = reinterpret_cast<T*>(base + used);
    used += (std::max<size_t>(count, 1) * sizeof(T) + 255) & ~(size_t)255;
  }
};

// The build's working memory: one block per device kept between builds (see build_bvh_on_device)
struct BuildCache {
  std::mutex mu;
  void* p[PT_MAX_DEVICES] = {};
  size_t bytes[PT_MAX_DEVICES] = {};
  bool busy[PT_MAX_DEVICES] = {};
};
BuildCache& build_cache() {
  static BuildCache c;
  return c;
}
struct BuildBlock {
  void* p = nullptr;
  int dev = -1;       // >= 0: p is the device's cached block
  bool own = false;   // p is a pool allocation of this build alone
  cudaError_t acquire(size_t bytes, cudaStream_t st) {
    int d = 0;
    cudaError_t e = cudaGetDevice(&d);
    if (e != cudaSuccess) return e;
    BuildCache& c = build_cache();
    {
      std::lock_guard<std::mutex> lock(c.mu);
      if (d >= 0 && d < PT_MAX_DEVICES && !c.busy[d]) {
        if (c.bytes[d] < bytes) {
          if (c.p[d]) cudaFreeAsync(c.p[d], st);
          c.p[d] = nullptr;
          c.bytes[d] = 0;
          e = pool_alloc(&c.p[d], bytes, st);
          if (e != cudaSuccess) return e;
          c.bytes[d] = bytes;
        }
        c.busy[d] = true;
        dev = d;
        p = c.p[d];
        return cudaSuccess;
      }
    }
    own = true;
    return pool_alloc(&p, bytes, st);
  }
  void release(cudaStream_t st) {
    if (own && p) cudaFreeAsync(p, st);
    if (dev >= 0) {
      cudaStreamSynchronize(st);  // the next build may run on another stream
      BuildCache& c = build_cache();
      std::lock_guard<std::mutex> lock(c.mu);
      c.busy[dev] = false;
    }
    p = nullptr;
    dev = -1;
    own = false;
  }
  ~BuildBlock() { release(0); }
};

}  // namespace

// ptrs_trim_memory: the cached working memory of the BVH builder goes back to the pool (and from there to the driver)
void release_bvh_build_cache() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= PT_MAX_DEVICES) return;
  BuildCache& c = build_cache();
  std::lock_guard<std::mutex> lock(c.mu);
  if (c.busy[d] || !c.p[d]) return;
  cudaFreeAsync(c.p[d], 0);
  c.p[d] = nullptr;
  c.bytes[d] = 0;
}

// Builds the BVH over n primitives given as device arrays in the caller's order.  On success *nodes_out holds
// *n_nodes_out 32-byte records (as float4 pairs) and *perm_out the primitive order (BVH position -> caller index);
// both are stream-ordered allocations the caller frees with cudaFreeAsync.  Returns a cudaError_t.
int build_bvh_on_device(cudaStream_t st, uint32_t n, const uint32_t* d_prim_vertex, const float* d_pos, float4** nodes_out, uint32_t* n_nodes_out,
                        uint32_t** perm_out, uint32_t* depth_out) {
  *nodes_out = nullptr;
  *perm_out = nullptr;
  *n_nodes_out = 0;
  *depth_out = 0;
  if (n == 0) return cudaSuccess;
  // tree topology: PLOC clustering; PTRS_BVH_BUILDER=lbvh selects the plain radix tree (a third of the build time,
  // 10 - 30 % slower to traverse: profiles/experiments/README.md)
  bool ploc = n > 1;
  if (const char* b = std::getenv("PTRS_BVH_BUILDER")) ploc = ploc && std::strcmp(b, "lbvh") != 0;
  const bool debug = std::getenv("PTRS_BVH_DEBUG") != nullptr;  // phase and round trace on stderr (synchronises between phases)
  auto t_phase = std::chrono::steady_clock::now();
  auto phase = [&](const char* what) {
    if (!debug) return;
    cudaStreamSynchronize(st);
    const auto t_now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "bvh build: %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t_now - t_phase).count());
    t_phase = t_now;
  };
  BuildArrays A{};
  uint64_t* keys_sorted = nullptr;
  uint32_t *perm_in = nullptr, *perm_sorted = nullptr, *perm_final = nullptr;
  uint32_t *cid_a = nullptr, *cid_b = nullptr, *cid_out = nullptr, *nn = nullptr, *keep = nullptr, *rank = nullptr, *cells = nullptr;
  void *sort_tmp = nullptr, *scan_tmp = nullptr;
  float4* nodes = nullptr;
  cudaError_t e = cudaSuccess;
  auto ok = [&](cudaError_t r) {
    if (e == cudaSuccess && r != cudaSuccess) e = r;
    return e == cudaSuccess;
  };
  const size_t n_int = n > 1 ? n - 1 : 0;
  size_t sort_bytes = 0;
  ok(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, A.keys, keys_sorted, perm_in, perm_sorted, (int)n, 0, 63, st));
  size_t scan_bytes = 0;
  if (ploc) ok(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, keep, rank, (int)n, st));
  // Working memory (190 B per primitive) comes from a per-device block the library keeps between builds (released by
  // ptrs_trim_memory): taken from the pool per build, a block of this size displaces the pool's cached blocks and the node
  // array allocated afterwards has to map fresh memory — 20 - 500 ms against the 17 ms the kernels of a 10 M-triangle
  // build take.  A second build running concurrently on the same device falls back to a block of its own.
  Arena arena;
  auto carve = [&](Arena& ar) {
    ar.take(&A.pb_min, n);
    ar.take(&A.pb_max, n);
    ar.take(&A.keys, n);
    ar.take(&perm_in, n);
    ar.take(&keys_sorted, n);
    char* tmp = nullptr;
    ar.take(&tmp, std::max<size_t>(sort_bytes, 16));
    sort_tmp = tmp;
    ar.take(&A.node, n_int);
    ar.take(&A.leaf_parent, n);
    ar.take(&A.box, 2 * (size_t)n);
    ar.take(&A.cbounds, 6);
    if (ploc) {
      ar.take(&cid_a, n);
      ar.take(&cid_b, n);
      ar.take(&cid_out, n);
      ar.take(&nn, n);
      ar.take(&keep, n);
      ar.take(&rank, n);
      ar.take(&cells, 2);  // [0] node-id counter, [1] length of the next cluster sequence
      char* tmp2 = nullptr;
      ar.take(&tmp2, std::max<size_t>(scan_bytes, 16));
      scan_tmp = tmp2;
      ar.take(&A.leaf_pos, n);
    }
  };
  carve(arena);  // sizes only
  BuildBlock block;
  ok(block.acquire(arena.used, st));
  ok(pool_alloc(reinterpret_cast<void**>(&perm_sorted), (size_t)n * 4, st));  // survives unless PLOC re-orders the primitives
  const int grid = 148 * 8;
  uint32_t n_interior_root = 0;
  phase("allocation");
  if (e == cudaSuccess) {
    arena = Arena{static_cast<char*>(block.p), 0};
    carve(arena);
    A.perm = perm_in;
    const uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    ok(cudaMemcpyAsync(A.cbounds, init, sizeof(init), cudaMemcpyHostToDevice, st));
    prim_bounds_kernel<<<grid, 256, 0, st>>>(d_prim_vertex, d_pos, n, A);
    morton_kernel<<<grid, 256, 0, st>>>(n, A);
    ok(cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, A.keys, keys_sorted, perm_in, perm_sorted, (int)n, 0, 63, st));
    A.perm = perm_sorted;
    A.keys = keys_sorted;
    phase("bounds, morton codes, sort");
    if (ploc) {
      ploc_init_kernel<<<grid, 256, 0, st>>>(n, A, cid_a);
      ok(cudaMemsetAsync(cells, 0, 8, st));
      uint32_t m = n, *cur = cid_a, *nxt = cid_b;
      int rounds = 0;
      auto t_prev = std::chrono::steady_clock::now();
      while (e == cudaSuccess && m > 1) {
        if (++rounds > PLOC_MAX_ROUNDS) {  // adversarial input (never seen: ~1.5 log2 n rounds): the radix tree is built instead
          ploc = false;
          break;
        }
        const int g = (int)std::min<uint32_t>((uint32_t)grid, (m + 255u) / 256u);
        ploc_nn_kernel<<<g, PLOC_BLOCK, 0, st>>>(m, cur, A.box, nn);
        ploc_merge_kernel<<<g, 256, 0, st>>>(m, n, cur, nn, A, cells, cid_out, keep);
        ok(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, keep, rank, (int)m, st));
        ploc_compact_kernel<<<g, 256, 0, st>>>(m, cid_out, keep, rank, nxt, cells + 1);
        uint32_t m_next = 0;
        ok(cudaMemcpyAsync(&m_next, cells + 1, 4, cudaMemcpyDeviceToHost, st));
        ok(cudaStreamSynchronize(st));
        ok(cudaGetLastError());
        if (e == cudaSuccess && (m_next == 0 || m_next >= m)) e = cudaErrorUnknown;  // every round merges at least one pair
        if (debug) {
          const auto t_now = std::chrono::steady_clock::now();
          std::fprintf(stderr, "ploc round %d: %u -> %u clusters, %.3f ms\n", rounds, m, m_next, std::chrono::duration<double, std::milli>(t_now - t_prev).count());
          t_prev = t_now;
        }
        m = m_next;
        std::swap(cur, nxt);
      }
      if (ploc) ok(cudaMemcpyAsync(&n_interior_root, &A.node[0].n_interior, 4, cudaMemcpyDeviceToHost, st));
    }
    if (!ploc && n > 1) {
      A.leaf_pos = nullptr;
      radix_tree_kernel<<<grid, 256, 0, st>>>(A.keys, (int)n, A);
      refit_kernel<<<grid, 256, 0, st>>>(n, A);
      ok(cudaMemcpyAsync(&n_interior_root, &A.node[0].n_interior, 4, cudaMemcpyDeviceToHost, st));
    }
    ok(cudaStreamSynchronize(st));
    ok(cudaGetLastError());
    phase("tree topology and boxes");
  }
  if (e == cudaSuccess && ploc && n_interior_root != 0) {
    ok(pool_alloc(reinterpret_cast<void**>(&perm_final), (size_t)n * 4, st));  // survives instead of the sorted order
    if (e == cudaSuccess) ploc_positions_kernel<<<grid, 256, 0, st>>>(n, A, perm_sorted, perm_final);
  } else {
    A.leaf_pos = nullptr;
  }
  if (e == cudaSuccess) {
    const uint32_t n_nodes = 2u + 2u * n_interior_root;
    ok(pool_alloc(reinterpret_cast<void**>(&nodes), (size_t)n_nodes * 32, st));
    if (e == cudaSuccess) {
      if (n_interior_root == 0) {
        single_leaf_kernel<<<1, 32, 0, st>>>(n, A, nodes);
      } else {
        // cbounds is dead after morton_kernel: its first word becomes the depth cell
        ok(cudaMemsetAsync(A.cbounds, 0, 4, st));
        emit_kernel<<<grid, 256, 0, st>>>(n, A, nodes, A.cbounds);
        ok(cudaMemcpyAsync(depth_out, A.cbounds, 4, cudaMemcpyDeviceToHost, st));
        ok(cudaStreamSynchronize(st));
      }
      ok(cudaGetLastError());
      *n_nodes_out = n_nodes;
    }
  }
  phase("positions, node emission");
  block.release(st);
  phase("free");
  if (e != cudaSuccess) {
    if (nodes) cudaFreeAsync(nodes, st);
    if (perm_sorted) cudaFreeAsync(perm_sorted, st);
    if (perm_final) cudaFreeAsync(perm_final, st);
    return (int)e;
  }
  *nodes_out = nodes;
  if (perm_final) {
    cudaFreeAsync(perm_sorted, st);
    *perm_out = perm_final;
  } else {
    *perm_out = perm_sorted;
  }
  return (int)cudaSuccess;
}

void launch_assemble_tris(cudaStream_t st, uint32_t n, const uint32_t* perm, const uint32_t* prim_vertex, const float* pos, const int32_t* prim_mesh,
                          const int32_t* prim_material, const int32_t* prim_area_light, const PtrsMesh* meshes, float4* tri_verts, uint4* tri_index,
                          uint32_t* inv_perm) {
  if (n == 0) return;
  assemble_tris_kernel<<<148 * 8, 256, 0, st>>>(n, perm, prim_vertex, pos, prim_mesh, prim_material, prim_area_light, meshes, tri_verts, tri_index, inv_perm);
}
// returns the error bits of validate_prims_kernel (0 = fine), or a negative cudaError_t
int validate_prims_on_device(cudaStream_t st, uint32_t n, const uint32_t* prim_vertex, const int32_t* prim_mesh, const int32_t* prim_material,
                             const int32_t* prim_area_light, uint32_t n_verts, uint32_t n_meshes, uint32_t n_materials, uint32_t n_lights,
                             const PtrsLight* lights) {
  if (n == 0) return 0;
  uint32_t* d_err = nullptr;
  cudaError_t e = pool_alloc(reinterpret_cast<void**>(&d_err), 4, st);
  if (e != cudaSuccess) return -(int)e;
  cudaMemsetAsync(d_err, 0, 4, st);
  validate_prims_kernel<<<148 * 8, 256, 0, st>>>(n, prim_vertex, prim_mesh, prim_material, prim_area_light, n_verts, n_meshes, n_materials, n_lights, lights, d_err);
  uint32_t h = 0;
  e = cudaMemcpyAsync(&h, d_err, 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFreeAsync(d_err, st);
  return e == cudaSuccess ? (int)h : -(int)e;
}

// d_raw: the n reference-order records on the device; *out receives 2 (n_interior + 1) records in the traversal layout
int pair_layout_on_device(cudaStream_t st, const float4* d_raw, uint32_t n, uint32_t n_interior, float4** out, uint32_t* n_out) {
  *out = nullptr;
  *n_out = 0;
  if (n == 0) return (int)cudaSuccess;
  const uint32_t n_dev = 2u * (n_interior + 1u);
  uint32_t *flag = nullptr, *rank = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flag, rank, (int)n, st);
  cudaError_t e = pool_alloc(reinterpret_cast<void**>(&flag), (size_t)n * 4, st);
  if (e == cudaSuccess) e = pool_alloc(reinterpret_cast<void**>(&rank), (size_t)n * 4, st);
  if (e == cudaSuccess) e = pool_alloc(&tmp, tmp_bytes ? tmp_bytes : 1, st);
  if (e == cudaSuccess) e = pool_alloc(reinterpret_cast<void**>(out), (size_t)n_dev * 32, st);
  if (e == cudaSuccess) {
    interior_flag_kernel<<<148 * 8, 256, 0, st>>>(d_raw, n, flag);
    e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, rank, (int)n, st);
  }
  if (e == cudaSuccess) {
    pair_layout_kernel<<<148 * 8, 256, 0, st>>>(d_raw, n, rank, *out);
    e = cudaGetLastError();
  }
  if (flag) cudaFreeAsync(flag, st);
  if (rank) cudaFreeAsync(rank, st);
  if (tmp) cudaFreeAsync(tmp, st);
  if (e != cudaSuccess && *out) {
    cudaFreeAsync(*out, st);
    *out = nullptr;
  }
  if (e == cudaSuccess) *n_out = n_dev;
  return (int)e;
}

void launch_remap_light_prims(cudaStream_t st, PtrsLight* lights, uint32_t n_lights, const uint32_t* inv_perm) {
  if (n_lights == 0) return;
  remap_light_prims_kernel<<<(n_lights + 127) / 128, 128, 0, st>>>(lights, n_lights, inv_perm);
}

}  // namespace ptrs
