// Host-callable launchers of the kernels, one group per translation unit.  Every launcher sizes its
// persistent grid as (resident CTAs per SM) x (SM count) from the occupancy API, cached per DEVICE
// (PT_GRID below): handles on different devices may be driven from different host threads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/ptrs_b200.h"

namespace ptrs {
struct DevScene;
struct PathArrays;
struct RoundCounters;
struct GlobalCounters;
struct RenderConst;

// ptrs_b200.cu: stream-ordered allocation from the library's private memory pool of the current device
cudaError_t pool_alloc(void** p, size_t bytes, cudaStream_t st);

// k_misc.cu
void launch_generate(cudaStream_t st, int sm, const RenderConst& rc, const uint32_t* sobol, const PathArrays& P, uint64_t work_base,
                     uint32_t n_work, const int* list_xy, const int* list_s, int* q_ext, RoundCounters* ctr);
void launch_shade_miss(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, const int* q, RoundCounters* ctr);
void launch_connect_resolve(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, const int* q_nee, RoundCounters* ctr);
void launch_accumulate(cudaStream_t st, int sm, const RenderConst& rc, const PathArrays& P, uint32_t n, float4* film);
void launch_gather_probe(cudaStream_t st, int sm, const float4* buf, size_t n_blocks64, int per_thread, uint32_t* sink, uint64_t* n_gathers);
void launch_read_probe(cudaStream_t st, int sm, const float4* buf, size_t n_pairs, int reps, uint32_t* sink);
void launch_build_guide(cudaStream_t st, const float* cdf, uint32_t size, uint32_t rows, uint32_t K, uint32_t* guide);
void launch_resolve(cudaStream_t st, const float4* film, uint32_t n, float* rgb, uint8_t* rgba8);
void launch_sobol_probe(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, const int* xy, const int* s, uint32_t n,
                        const int* dims, uint32_t n_dims, float* out, uint64_t* out_index, int generic);
void launch_sobol_split_build(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, uint32_t* tab);
void launch_ray_probe(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, const int* xy, const int* s, uint32_t n, PtrsRay* rays,
                      float* p_film, float* rxry);

// k_trace.cu
void launch_extend(cudaStream_t st, int sm, bool count, const DevScene& sc, const PathArrays& P, const int* q_ext, int* q_class, uint32_t cap,
                   RoundCounters* ctr, GlobalCounters* g);
void launch_connect(cudaStream_t st, int sm, bool count, const DevScene& sc, const PathArrays& P, uint32_t cap, bool closest_only, RoundCounters* ctr,
                    GlobalCounters* g);
void launch_occlusion(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, RoundCounters* ctr, GlobalCounters* g);
void launch_intersect(cudaStream_t st, int sm, bool any_hit, bool count, const DevScene& sc, const PtrsRay* rays, uint32_t n, PtrsHit* hits,
                      uint8_t* occluded, uint32_t* ticket, GlobalCounters* g, const uint32_t* prim_map);

// k_tables.cu: MIP pyramid levels, env-light density and Distribution1D rows built on the device
void launch_mip_level(cudaStream_t st, const float* prev, int pw, int ph, int channels, int wrap, float* out, int sres, int tres);
void launch_pack_shading(cudaStream_t st, uint32_t n, const float4* tri_verts, const uint4* tri_index, const float* normal, const float* uv, float4* out);
void launch_env_density(cudaStream_t st, const DevScene& sc, int mip, int nu, int nv, const float* row_sin, int mode, int il, float delta, float* func);
void launch_row_cdf(cudaStream_t st, const float* func, int n, int rows, float* cdf, float* func_int);

// k_bvh.cu
void release_bvh_build_cache();  // k_bvh.cu: the builder's cached working memory of the current device
int build_bvh_on_device(cudaStream_t st, uint32_t n, const uint32_t* d_prim_vertex, const float* d_pos, float4** nodes_out, uint32_t* n_nodes_out,
                        uint32_t** perm_out, uint32_t* depth_out);
void launch_assemble_tris(cudaStream_t st, uint32_t n, const uint32_t* perm, const uint32_t* prim_vertex, const float* pos, const int32_t* prim_mesh,
                          const int32_t* prim_material, const int32_t* prim_area_light, const PtrsMesh* meshes, float4* tri_verts, uint4* tri_index,
                          uint32_t* inv_perm);
int validate_prims_on_device(cudaStream_t st, uint32_t n, const uint32_t* prim_vertex, const int32_t* prim_mesh, const int32_t* prim_material,
                             const int32_t* prim_area_light, uint32_t n_verts, uint32_t n_meshes, uint32_t n_materials, uint32_t n_lights,
                             const PtrsLight* lights);
int pair_layout_on_device(cudaStream_t st, const float4* d_raw, uint32_t n, uint32_t n_interior, float4** out, uint32_t* n_out);
void launch_remap_light_prims(cudaStream_t st, PtrsLight* lights, uint32_t n_lights, const uint32_t* inv_perm);

// k_sah.cu: the reference's SAH tree (ptrs_host::build_bvh) built on the device, bit for bit
int build_sah_bvh_on_device(cudaStream_t st, uint32_t n, const uint32_t* d_prim_vertex, const float* d_pos, int max_prims, uint32_t depth_limit,
                            float4** nodes_out, uint32_t* n_nodes_out, uint32_t** perm_out, uint32_t* max_depth_out);

// k_probe.cu, built twice (shade-kernel arithmetic / exact arithmetic)
#define PT_DECL_PROBES(SUF)                                                                                                                       \
  void launch_bxdf_eval_probe_##SUF(cudaStream_t st, const PtrsLobeDesc& d, const float* wo, const float* wi, uint32_t n, float* out);             \
  void launch_bxdf_sample_probe_##SUF(cudaStream_t st, const PtrsLobeDesc& d, const float* wo, const float* u, uint32_t n, float* out);            \
  void launch_light_sample_probe_##SUF(cudaStream_t st, const DevScene& sc, int light, const float* p, const float* nn, const float* u, uint32_t n, \
                                       float* out);                                                                                               \
  void launch_light_pdf_probe_##SUF(cudaStream_t st, const DevScene& sc, int light, const float* p, const float* nn, const float* wi, uint32_t n,  \
                                    float* out);
PT_DECL_PROBES(fast) PT_DECL_PROBES(exact)
#undef PT_DECL_PROBES

// k_shade.cu, built once per PtrsMaterialType
#define PT_DECL_SHADE(M)                                                                                                              \
  void launch_shade_##M(cudaStream_t st, int sm, const RenderConst& rc, const DevScene& sc, const PathArrays& P, const int* q, const float4* q_hit, \
                        int* q_next, int* q_nee, RoundCounters* ctr, RoundCounters* ctr_next);
PT_DECL_SHADE(0) PT_DECL_SHADE(1) PT_DECL_SHADE(2) PT_DECL_SHADE(3) PT_DECL_SHADE(4) PT_DECL_SHADE(5)
// the same kernels from translation units built with IEEE division / square root and no FMA contraction
PT_DECL_SHADE(exact_0) PT_DECL_SHADE(exact_1) PT_DECL_SHADE(exact_2) PT_DECL_SHADE(exact_3) PT_DECL_SHADE(exact_4) PT_DECL_SHADE(exact_5)
#undef PT_DECL_SHADE

#define PT_MAX_DEVICES 64
// resident CTAs per SM of `kernel` on the current device, looked up once per device (lock-free: a racing second
// lookup stores the same value)
template <class K>
inline int persistent_grid(std::atomic<int>* per_device, K kernel, int block, int sm_count, size_t smem = 0) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= PT_MAX_DEVICES) dev = 0;
  int per_sm = per_device[dev].load(std::memory_order_relaxed);
  if (per_sm == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    per_device[dev].store(per_sm, std::memory_order_relaxed);
  }
  return sm_count * per_sm;
}
// one cache per call site (the lambda's static is unique to it)
#define PT_GRID(kernel, block, sm)                       \
  ([&]() {                                               \
    static std::atomic<int> cache__[PT_MAX_DEVICES];     \
    return persistent_grid(cache__, kernel, block, sm);  \
  }())
}  // namespace ptrs
