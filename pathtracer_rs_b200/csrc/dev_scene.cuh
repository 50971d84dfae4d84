// Device-resident scene: the PtrsSceneDesc re-laid-out for 128-bit loads.
//   nodes      32 B records identical to the reference's LinearBVHNode, read as two float4 via the
//              non-coherent path (ld.global.nc.v4)
//   tri_verts  48 B per primitive = 3 x float4: xyz = vertex k, w = {material id, area-light id,
//              mesh flags | alpha texture} as raw bits.  The 36 algorithmic bytes + 12 B of shading
//              metadata that would otherwise be a second dependent load.
//   tri_index  16 B per primitive: three global vertex indices + mesh id, only read by shading.
//   tri_shade  64 B per primitive: the three shading normals and uvs of the triangle, gathered once at scene creation
//              so that shading reads them with two 32-byte loads that depend on the primitive id alone.
#pragma once
#include "../../include/ptrs_b200.h"
#include "dev_math.cuh"

namespace ptrs {

struct DevEnv {
  float light_to_world[16];
  float world_to_light[16];
  int mip, nu, nv, pad;
  const float* cond_func;
  const float* cond_cdf;
  const float* cond_func_int;
  const float* marg_func;
  const float* marg_cdf;
  float marg_func_int;
  float pad2;
  // guide tables (built on the device at scene creation): guide[k] = number of cdf entries <= k / K, K a power
  // of two >= n.  They bracket find_interval's partition point for any u in [k/K, (k+1)/K), so the binary
  // search of math.rs:186-201 runs over (on average) one element instead of n; same result.
  const uint32_t* cond_guide;  // nv rows x (ku + 1)
  const uint32_t* marg_guide;  // kv + 1
  uint32_t ku, kv;
};

struct DevScene {
  const float4* nodes;      // 2 per node
  const float4* tri_verts;  // 3 per prim
  const uint4* tri_index;   // 1 per prim
  const float4* tri_shade;  // 4 per prim: shading normals n0 n1 n2 (9 floats), uvs (6 floats, the defaults of shape.rs:34-48 when the mesh has none), 1 spare
  const float* normal;
  const float* tangent;
  const float* uv;
  const PtrsMesh* meshes;
  const PtrsMaterial* materials;
  const PtrsTexture* textures;
  const PtrsMipMap* mipmaps;
  const float* texels;
  const PtrsLight* lights;
  const int* infinite_lights;
  const DevEnv* envs;
  const uint32_t* sobol;    // SOBOL_MATRICES_32, 1024 dimensions x 52 columns
  const uint32_t* sobol_t;  // the same table bit-major: 52 x 1024
  uint32_t n_nodes, n_prims, n_lights, n_infinite_lights;
  uint32_t box_min;    // traversal scheduling threshold, see trace_fast
  uint32_t pop_twice;  // traversal scheduling: a second pop when the first one leaves the lane without a node (trees beyond L1 size)
  uint32_t dist_order;  // library-built tree: of two entered children the one with the smaller entry distance is visited first
  // 1 when some material parameter or normal map is an image texture: the only consumer of the camera-ray
  // differentials (MIPMap::lookup's filter width, texture.rs:431-445).  Without one, shade skips
  // compute_differentials — every value it would produce is unread.
  uint32_t uses_differentials;
  // occlusion tree (any-hit rays only, trace_occlusion): 128-byte wide nodes collapsed from the reference-built tree, 8
  // float4 per node; n_wnodes == 0 when the scene has none (device-built tree, or a tree the collapse does not accept)
  const float4* wnodes;
  uint32_t n_wnodes;
};

// tri_verts[3 * prim + 2].w packs: bits 0..7 mesh flags, bit 8 has-alpha, bits 9.. alpha texture id
#define PT_TRI_ALPHA_BIT 0x100u

struct DevRay {
  V3 o, d;
  float t_max;
};

struct DevHit {
  int prim;
  float t, b0, b1, b2;
};

}  // namespace ptrs
