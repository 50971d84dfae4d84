/*
 * ptrs_b200.h — C ABI of the B200-native rendering hot path for pathtracer-rs.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI layer today: its path
 * integrator is called in-process as
 *     PathIntegrator::new(log, sampler_builder, max_depth, progress)   src/pathtracer/integrator.rs:230
 *     PathIntegrator::preprocess(&RenderScene)                         src/pathtracer/integrator.rs:250
 *     PathIntegrator::render(&self, &Camera, &RenderScene)             src/pathtracer/integrator.rs:536
 *     RenderScene::{intersect, intersect_p, world_bound}               src/pathtracer/mod.rs:92-102
 *     Film::{clear, get_sample_bounds, to_rgba_image, ...}             src/common/film.rs:164-271
 * and its own (stub) GPU hook sits at OptixAccelerator::new(&RenderScene)/intersect()
 * (src/pathtracer/gpu/optix.rs:160,292).  The entry points below are what a Rust `extern "C"` block
 * built from build.rs (build.rs:14-36 is where the reference shells out to nvcc) would bind; the
 * binding stub is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C, POD structs, explicit sizes; no exceptions or aborts cross the boundary
 *   - every call returns int32_t: PTRS_OK (0) or a negative PtrsStatus; ptrs_last_error() gives a
 *     thread-local message for the last failing call
 *   - host pointers unless the name says `_device`; `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream)
 *   - a scene handle owns device copies of everything in the PtrsSceneDesc (the caller may free its
 *     buffers as soon as ptrs_scene_create returns); a handle is not re-entrant
 *   - there is no CPU fallback: with no usable CUDA device every call fails with PTRS_ERR_CUDA
 */
#ifndef PTRS_B200_H
#define PTRS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTRS_ABI_VERSION 1
#define PTRS_COMM_ID_BYTES 128 /* size of the communicator id ptrs_comm_unique_id hands out (ncclUniqueId) */

typedef enum PtrsStatus {
  PTRS_OK = 0,
  PTRS_ERR_INVALID_ARGUMENT = -1,
  PTRS_ERR_CUDA = -2,
  PTRS_ERR_UNSUPPORTED = -3,
  PTRS_ERR_OUT_OF_MEMORY = -4,
  PTRS_ERR_NCCL = -5
} PtrsStatus;

/* ------------------------------------------------------------------------------------------------
 * Accelerator records
 * ---------------------------------------------------------------------------------------------- */

/* Ray {o, d, t_max}: src/common/ray.rs:2-6 (28 bytes). */
typedef struct PtrsRay {
  float o[3];
  float d[3];
  float t_max;
} PtrsRay;

/* What the integrator keeps of a closest hit: the primitive (index into the BVH-ordered primitive
 * array, -1 = miss), the parametric distance and the barycentrics of Triangle::intersect
 * (src/pathtracer/shape.rs:156-161).  Everything else in SurfaceMediumInteraction is a pure
 * function of these and the ray. */
typedef struct PtrsHit {
  int32_t prim;
  float t;
  float b0, b1, b2;
} PtrsHit;

/* LinearBVHNode, #[repr(C, align(32))]: src/pathtracer/accelerator.rs:83-95.
 * offset = primitives_offset for a leaf (n_prims > 0) / second_child_offset for an interior node;
 * the first child of an interior node is the next node in the array. */
typedef struct PtrsBvhNode {
  float bounds_min[3];
  float bounds_max[3];
  uint32_t offset;
  uint16_t n_prims;
  uint8_t axis;
  uint8_t pad;
} PtrsBvhNode;

/* ------------------------------------------------------------------------------------------------
 * Scene description (what RenderScene holds after the importers ran, flattened)
 * ---------------------------------------------------------------------------------------------- */

/* TriangleMesh attribute presence: src/pathtracer/shape.rs:581-589 (`normal`, `s`, `uv` may be
 * empty Vecs; `alpha_mask` is an Option). */
enum {
  PTRS_MESH_HAS_NORMAL = 1,
  PTRS_MESH_HAS_TANGENT = 2,
  PTRS_MESH_HAS_UV = 4
};

typedef struct PtrsMesh {
  uint32_t flags;
  int32_t alpha_tex; /* float texture id or -1 (shape.rs:228-244, 471-521) */
} PtrsMesh;

/* Texture<T>: src/pathtracer/texture.rs.  `channels` is 1 for f32 and 3 for Spectrum / Vector3. */
typedef enum PtrsTextureType {
  PTRS_TEX_CONSTANT = 0, /* texture.rs:15-29   value = v1 */
  PTRS_TEX_CHECKER = 1,  /* texture.rs:56-89   v1, v2, UVMap */
  PTRS_TEX_IMAGE = 2     /* texture.rs:91-192  MIPMap + UVMap */
} PtrsTextureType;

typedef enum PtrsWrapMode { /* src/common/mod.rs:64-69 */
  PTRS_WRAP_REPEAT = 0,
  PTRS_WRAP_BLACK = 1,
  PTRS_WRAP_CLAMP = 2
} PtrsWrapMode;

typedef struct PtrsTexture {
  int32_t type;
  int32_t channels;
  float v1[3];
  float v2[3];
  float su, sv, du, dv; /* UVMap: texture.rs:31-54 */
  int32_t mip;          /* index into mipmaps, -1 if none */
  int32_t pad;
} PtrsTexture;

/* MIPMap pyramid as built by MIPMap::new (texture.rs:279-405), already resampled to powers of two
 * and box-filtered by the host.  Level l is `height[l]` rows of `width[l]` texels of `channels`
 * floats, row-major, starting at texels[level_offset[l]] (offset counted in floats).
 * A description may instead carry LEVEL 0 ONLY (n_levels == 1 for an image larger than one texel, both
 * extents powers of two): ptrs_scene_create then builds the box-filtered levels on the device
 * (texture.rs:345-405), bit-identical to the host's. */
#define PTRS_MAX_MIP_LEVELS 16
typedef struct PtrsMipMap {
  int32_t channels;
  int32_t wrap;
  int32_t n_levels;
  int32_t width[PTRS_MAX_MIP_LEVELS];
  int32_t height[PTRS_MAX_MIP_LEVELS];
  uint64_t level_offset[PTRS_MAX_MIP_LEVELS];
} PtrsMipMap;

/* Material enum: src/pathtracer/material/mod.rs:28-37.  tex[] meaning by type:
 *   MATTE      kd                                            (mod.rs:155-167)
 *   MIRROR     -                                             (mod.rs:180-195)
 *   GLASS      kr, kt, index                                 (mod.rs:216-255)
 *   METAL      eta, k, r, u_roughness, v_roughness           (metal.rs:49-93)
 *   SUBSTRATE  kd, ks, nu, nv                                (substrate.rs:42-68)
 *   DISNEY     color, metallic, eta, roughness               (disney.rs:172-263)
 * normal_map >= 0 wraps the material in Material::Normal (mod.rs:39-79, 130-135). */
typedef enum PtrsMaterialType {
  PTRS_MAT_MATTE = 0,
  PTRS_MAT_MIRROR = 1,
  PTRS_MAT_GLASS = 2,
  PTRS_MAT_METAL = 3,
  PTRS_MAT_SUBSTRATE = 4,
  PTRS_MAT_DISNEY = 5,
  PTRS_MAT_COUNT = 6
} PtrsMaterialType;

typedef struct PtrsMaterial {
  int32_t type;
  int32_t normal_map;      /* Vector3 texture id or -1 */
  int32_t tex[5];
  int32_t remap_roughness; /* metal.rs:75-78, substrate.rs:56-59 */
} PtrsMaterial;

/* Lights: src/pathtracer/light.rs. */
typedef enum PtrsLightType {
  PTRS_LIGHT_POINT = 0,       /* light.rs:86-150   pos = p_light, color = I */
  PTRS_LIGHT_DIRECTIONAL = 1, /* light.rs:152-229  pos = w_light (normalised), color = L */
  PTRS_LIGHT_AREA = 2,        /* light.rs:231-319  one per emissive triangle; prim, ke_tex, area */
  PTRS_LIGHT_INFINITE = 3     /* light.rs:321-503  env */
} PtrsLightType;

typedef struct PtrsLight {
  int32_t type;
  int32_t prim;   /* AREA: index into the BVH-ordered primitive array */
  int32_t ke_tex; /* AREA: Spectrum texture id (emission map) */
  int32_t env;    /* INFINITE: index into envs */
  float pos[3];
  float color[3];
  float area;            /* AREA: Triangle::area(), shape.rs:533-539 */
  float world_radius;    /* DIRECTIONAL / INFINITE: Light::preprocess, bounds.rs:126-134 */
  float world_center[3];
  float pad;
} PtrsLight;

/* InfiniteAreaLight state: light.rs:321-399.  The Distribution2D (sampling.rs:185-230) is passed
 * exactly as the reference builds it: nv conditional rows of nu entries.
 * With all five array pointers NULL the library tabulates the density from the environment map and builds
 * the distribution on the device (light.rs:372-387, sampling.rs:133-162, 185-209), bit-identical to the
 * host's; nu / nv <= 0 then default to twice the map's resolution (light.rs:375-376). */
typedef struct PtrsEnvLight {
  float light_to_world[16]; /* row-major 4x4, Projective3 */
  float world_to_light[16];
  int32_t mip;              /* Spectrum MIPMap id (WrapMode::Repeat) */
  int32_t nu, nv;
  int32_t pad;
  const float* cond_func;     /* nv * nu        */
  const float* cond_cdf;      /* nv * (nu + 1)  */
  const float* cond_func_int; /* nv             */
  const float* marg_func;     /* nv  (== cond_func_int) */
  const float* marg_cdf;      /* nv + 1         */
  float marg_func_int;
  float pad2;
} PtrsEnvLight;

typedef struct PtrsSceneDesc {
  uint32_t abi_version; /* PTRS_ABI_VERSION */

  /* accelerator: BVH::nodes / BVH::primitives (accelerator.rs:97-100) in the reference's order */
  uint32_t n_nodes;
  const PtrsBvhNode* nodes;
  uint32_t n_prims;
  const uint32_t* prim_vertex; /* 3 * n_prims global vertex indices (Triangle::indices + mesh base) */
  const int32_t* prim_mesh;    /* n_prims */
  const int32_t* prim_material;
  const int32_t* prim_area_light; /* light id or -1 (GeometricPrimitive::area_light) */

  /* vertex pools; normal / tangent / uv may be NULL when no mesh uses them */
  uint32_t n_verts;
  const float* pos;     /* 3 * n_verts, world space (shape.rs:602-604) */
  const float* normal;  /* 3 * n_verts */
  const float* tangent; /* 3 * n_verts (TriangleMesh::s) */
  const float* uv;      /* 2 * n_verts */

  uint32_t n_meshes;
  const PtrsMesh* meshes;
  uint32_t n_materials;
  const PtrsMaterial* materials;
  uint32_t n_textures;
  const PtrsTexture* textures;
  uint32_t n_mipmaps;
  const PtrsMipMap* mipmaps;
  uint64_t n_texels; /* floats */
  const float* texels;

  /* RenderScene::lights / infinite_lights (src/pathtracer/mod.rs:84-89) */
  uint32_t n_lights;
  const PtrsLight* lights;
  uint32_t n_infinite_lights;
  const int32_t* infinite_lights; /* light ids */
  uint32_t n_envs;
  const PtrsEnvLight* envs;
} PtrsSceneDesc;

/* ------------------------------------------------------------------------------------------------
 * Camera, sampler and integrator settings
 * ---------------------------------------------------------------------------------------------- */

/* Camera: src/common/mod.rs:19-62.  The host builds it (Camera::new); the fields are the ones
 * generate_ray_differential reads (src/pathtracer/mod.rs:59-81). */
typedef struct PtrsCamera {
  float rot[4];   /* cam_to_world rotation, unit quaternion (i, j, k, w) */
  float trans[3]; /* cam_to_world translation */
  float pad0;
  float raster_to_screen[16]; /* row-major Affine3 */
  float persp[4];             /* Perspective3 m00, m11, m22, m23 */
  float dx_camera[3];
  float dy_camera[3];
  int32_t width, height; /* film resolution */
} PtrsCamera;

#define PTRS_FILTER_TABLE_WIDTH 16 /* src/common/film.rs:121 */

/* PathIntegrator fields (integrator.rs:219-246), SobolSamplerBuilder (sampler/sobol.rs:35-62) and
 * the film filter (film.rs:132-163, filter.rs:61-89).  Defaults = ptrs_render_params_default(). */
typedef struct PtrsRenderParams {
  int32_t spp;       /* samples per pixel as given; rounded up to a power of two like sobol.rs:37 */
  int32_t max_depth; /* main.rs default 15 */
  float rr_threshold; /* 1.0 */
  int32_t rr_start_depth; /* 3 */
  int32_t rr_enable;      /* 1 */
  /* sharding (not in the reference): render Sobol sample numbers s with
   * sample_begin <= s < sample_end and (s % sample_stride) == sample_phase */
  int32_t sample_begin, sample_end; /* end <= 0 means "all spp" */
  int32_t sample_stride, sample_phase; /* 1, 0 */
  float filter_radius[2];                                                 /* 2, 2 */
  float filter_table[PTRS_FILTER_TABLE_WIDTH * PTRS_FILTER_TABLE_WIDTH]; /* film.rs:135-144 */
  int32_t paths_per_batch; /* 0 = library default; wavefront batch size */
  int32_t flags;           /* PTRS_RENDER_* */
} PtrsRenderParams;

/* PtrsRenderParams.flags.  The traversal, sampler and camera kernels are always built with IEEE division / square
 * root and without FMA contraction (that is what makes hits, rays and Sobol draws bit-identical to the CPU path);
 * the shade kernels are by default built with contraction and the 2-ulp division / square root.
 * PTRS_RENDER_EXACT_SHADING selects shade kernels built like the rest — the parity mode: what still differs from
 * the reference is then its libm (sin, cos, atan2, acos, exp, ln, log2, pow) and nothing else. */
#define PTRS_RENDER_EXACT_SHADING 1

/* Counters of the last render on a scene handle. */
typedef struct PtrsStats {
  uint64_t camera_paths;
  uint64_t extension_rays; /* closest-hit rays of the main path (integrator.rs:416) */
  uint64_t shadow_rays;    /* any-hit rays (light.rs:39-41) */
  uint64_t mis_rays;       /* closest-hit rays of estimate_direct's BSDF sample (integrator.rs:119) */
  /* BVH nodes / triangles tested; filled only when ptrs_set_stats_mode(scene, 1) is on */
  uint64_t nodes_tested;     /* by the extend kernel (extension rays) */
  uint64_t tris_tested;
  uint64_t nee_nodes_tested; /* by the connect kernel (shadow + MIS rays) */
  uint64_t nee_tris_tested;
  float ms_generate, ms_extend, ms_shade, ms_shadow, ms_accumulate, ms_total;
  uint32_t launches; /* kernels launched by the last call */
  uint32_t batches;
  uint32_t extend_launches, connect_launches;
  /* ms_shadow split into its two kernels: connect_kernel (shadow + MIS ray traversal) and connect_resolve_kernel */
  float ms_connect_trace, ms_resolve;
} PtrsStats;

typedef struct PtrsScene PtrsScene; /* opaque */
typedef struct PtrsFilm PtrsFilm;   /* opaque: W x H x (r, g, b, weight) f32 on the device */
typedef struct PtrsComm PtrsComm;   /* opaque: one rank of an NCCL communicator over the GPUs that share a film */
typedef struct PtrsMultiScene PtrsMultiScene; /* opaque: one scene replica, film and stream per device, one process */

/* ------------------------------------------------------------------------------------------------
 * Entry points
 * ---------------------------------------------------------------------------------------------- */

/* library / device */
int32_t ptrs_abi_version(void);
const char* ptrs_last_error(void);
int32_t ptrs_device_count(int32_t* count);
int32_t ptrs_set_device(int32_t device); /* device used by handles created afterwards on this thread */

/* RenderScene construction / teardown (replaces holding Box<BVH> + lights in RenderScene) */
int32_t ptrs_scene_create(const PtrsSceneDesc* desc, PtrsScene** out);
/* Same, but the accelerator is built on the device (replaces the host-side BVH::new, accelerator.rs:103-346, when
 * start-up time matters: Morton order + PLOC clustering by merged surface area, leaves of at most 4 primitives — 16 ms
 * for 10 M triangles, and a tree that traverses as fast as or faster than the reference builder's on the scenes
 * measured; the environment variable PTRS_BVH_BUILDER=lbvh selects a plain radix tree).  desc->nodes / n_nodes are ignored and the
 * primitive arrays may be in any order; PtrsLight.prim and the prim ids reported by ptrs_intersect* refer to the
 * caller's order.  Closest hits (t, barycentrics) are those of ptrs_scene_create on the same geometry; only the
 * traversal cost and the winner among hits within an ulp of each other can differ (the reference's traversal
 * resolves those by visit order). */
int32_t ptrs_scene_create_device_bvh(const PtrsSceneDesc* desc, PtrsScene** out);
/* Same, but the accelerator is the reference's own: BVH::new(prims, max_prims_in_node) (accelerator.rs:103-346) built
 * on the device.  The tree equals the one BVH::new builds over the primitives in the order given, record for record
 * and in its primitive order, so hits (prim, t, barycentrics), traversal counters and any-hit answers equal those of
 * ptrs_scene_create over that tree, bit for bit.  desc->nodes / n_nodes are ignored; PtrsLight.prim and the prim ids
 * reported by ptrs_intersect* refer to the caller's order.  max_prims_in_node: 1 .. 65535 (the importers use 4).
 * A tree deeper than the 64-entry traversal stack is refused with PTRS_ERR_UNSUPPORTED, as by ptrs_scene_create. */
int32_t ptrs_scene_create_sah_bvh(const PtrsSceneDesc* desc, int32_t max_prims_in_node, PtrsScene** out);
/* node count of the device-side tree (any constructor) and the device build time (0 for a host-built BVH) */
int32_t ptrs_scene_bvh_info(const PtrsScene* scene, uint32_t* n_nodes, float* device_build_ms);
/* The device-side tree for inspection: 32-byte LinearBVHNode records in the traversal layout (root in slot 0, slot 1
 * unused, the two children of an interior node at offset and offset + 1); prim_order (optional, device-built trees
 * only) maps BVH primitive positions to the caller's primitive indices. */
int32_t ptrs_scene_download_nodes(const PtrsScene* scene, PtrsBvhNode* nodes, uint32_t capacity, uint32_t* prim_order);
/* The texture tables as the device holds them (pyramids completed by the library included): headers, pool size in
 * floats, and — if `texels` is not NULL — the pool itself; and an env light's Distribution2D (any array may be NULL). */
int32_t ptrs_scene_download_mipmaps(const PtrsScene* scene, PtrsMipMap* mipmaps, uint32_t capacity, uint64_t* n_texels,
                                    float* texels, uint64_t texel_capacity);
int32_t ptrs_scene_download_env(const PtrsScene* scene, int32_t env, int32_t* nu, int32_t* nv, float* cond_func,
                                float* cond_cdf, float* cond_func_int, float* marg_cdf, float* marg_func_int);
int32_t ptrs_scene_destroy(PtrsScene* scene);
int32_t ptrs_scene_world_bound(const PtrsScene* scene, float out_min_max[6]); /* mod.rs:100-102 */
uint64_t ptrs_scene_device_bytes(const PtrsScene* scene);
/* Device memory of destroyed scenes / films / path workspaces stays reserved in the device's default memory pool
 * for re-use by the next ptrs_scene_create / ptrs_render; this returns it to the driver. */
int32_t ptrs_trim_memory(void);
/* Diagnostic: read bandwidth of `reps` streaming passes (256-bit non-coherent loads, persistent grid) over a
 * zeroed device buffer of `bytes`.  A buffer that fits in L2 gives the L2 read bandwidth the traversal
 * kernels' roofline fraction is quoted against when the tree is cache resident; a much larger one the HBM
 * read bandwidth. */
int32_t ptrs_read_bandwidth(size_t bytes, int32_t reps, float* gb_per_s);
/* Same for the traversal's access pattern: independent 64-byte gathers at pseudo-random aligned positions of the
 * buffer, `gathers_per_thread` per thread of a persistent grid. */
int32_t ptrs_gather_bandwidth(size_t bytes, int32_t gathers_per_thread, float* gb_per_s);

/* RenderScene::intersect / intersect_p over a batch (mod.rs:92-98; accelerator.rs:359-475).
 * Host-buffer forms copy in and out; *_device forms take device pointers and only enqueue. */
int32_t ptrs_intersect(PtrsScene* scene, const PtrsRay* rays, size_t n, PtrsHit* hits);
int32_t ptrs_intersect_p(PtrsScene* scene, const PtrsRay* rays, size_t n, uint8_t* occluded);
int32_t ptrs_intersect_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n, PtrsHit* d_hits,
                              void* stream);
int32_t ptrs_intersect_p_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n,
                                uint8_t* d_occluded, void* stream);
/* same traversal with node / triangle test counters (roofline bookkeeping, SURVEY.md §8d) */
int32_t ptrs_intersect_counted_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n,
                                      PtrsHit* d_hits, int32_t any_hit, uint8_t* d_occluded,
                                      uint64_t* nodes_tested, uint64_t* tris_tested, void* stream);

/* Film (film.rs) */
int32_t ptrs_film_create(int32_t width, int32_t height, PtrsFilm** out);
int32_t ptrs_film_wrap_device(int32_t width, int32_t height, float* d_rgbw, PtrsFilm** out);
int32_t ptrs_film_destroy(PtrsFilm* film);
int32_t ptrs_film_clear(PtrsFilm* film, void* stream);                    /* film.rs:164-172 */
int32_t ptrs_film_download(PtrsFilm* film, float* rgbw /* W*H*4 */);       /* raw sums */
int32_t ptrs_film_resolve(PtrsFilm* film, float* rgb /* W*H*3 */);         /* film.rs:253-271 */
int32_t ptrs_film_resolve_srgb8(PtrsFilm* film, uint8_t* rgba /* W*H*4 */); /* film.rs:230-251 */
float* ptrs_film_device_ptr(PtrsFilm* film);
int32_t ptrs_film_sample_bounds(int32_t width, int32_t height, const float filter_radius[2],
                                int32_t out_min_max[4]); /* film.rs:174-185 */
/* The sample rectangle that completes a pixel crop: the smallest rectangle of sample positions ({x0, y0, x1, y1},
 * half-open, in the coordinates of ptrs_film_sample_bounds) whose samples include every contribution any pixel of
 * pixel_rect (half-open, inside the film) receives in a full render, clipped to the sample bounds.  Derived from the
 * float expressions of the film splat; for radius 2 it is pixel_rect grown by 2 on each side.  Host arithmetic only. */
int32_t ptrs_film_region_sample_rect(int32_t width, int32_t height, const float filter_radius[2], const int32_t pixel_rect[4],
                                     int32_t sample_rect[4]);

/* PathIntegrator */
int32_t ptrs_render_params_default(PtrsRenderParams* params); /* integrator.rs:237-245 + Gaussian */
int32_t ptrs_render(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params,
                    PtrsFilm* film, void* stream); /* integrator.rs:536; accumulates into film */
/* ptrs_render restricted to a rectangle of sample positions: sample_rect = {x0, y0, x1, y1}, half-open, a non-empty
 * rectangle inside ptrs_film_sample_bounds (so it may start at -2).  Every selected sample number (spp, sample range,
 * stride / phase) of every position inside it is traced, with the same Sobol index as in the full render, and splatted
 * into the full-size film; only film pixels within the filter footprint of the rectangle change.  Rectangles that
 * partition the sample bounds sum to the full render (integrator.rs:545-637 renders 16x16 tiles of them).
 * ptrs_stats counts camera_paths = area x selected samples.  ptrs_render is this call with the whole sample bounds. */
int32_t ptrs_render_region(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t sample_rect[4],
                           PtrsFilm* film, void* stream);
/* li() of integrator.rs:579 for chosen (pixel, sample number) pairs: out_rgb[3 i ..] = radiance of that
 * camera path.  Same kernels as ptrs_render with the film splat left out; parity probe. */
int32_t ptrs_path_radiance(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params,
                           const int32_t* pixels_xy, const int32_t* sample_nums, size_t n, float* out_rgb);
int32_t ptrs_stats(const PtrsScene* scene, PtrsStats* out);
int32_t ptrs_set_stats_mode(PtrsScene* scene, int32_t count_visits); /* counted traversal in render */

/* ------------------------------------------------------------------------------------------------
 * Several GPUs of one node (SURVEY.md §8e).  The reference parallelises PathIntegrator::render over
 * 16x16 tiles with rayon and merges tiles into the one film under a lock (integrator.rs:617-637,
 * film.rs:213-228); across GPUs the scene is replicated, the Sobol sample numbers of every pixel are
 * dealt round-robin (device g of N renders s = g (mod N); the global Sobol index is a pure function
 * of (pixel, sample number), sampler/sobol.rs:169-175) and the additive films are summed with ONE
 * NCCL reduce over NVLink.  The result equals the single-GPU film up to float summation order.
 * NCCL is loaded at run time (libnccl.so.2, or the file named by PTRS_NCCL_LIB); without it these
 * calls fail with PTRS_ERR_NCCL and everything else keeps working.
 * ---------------------------------------------------------------------------------------------- */

/* (a) one process, N devices: the library runs one host thread, stream, scene replica and film per
 * device (ncclCommInitAll).  devices == NULL means devices 0 .. n_devices-1; device_bvh != 0 builds
 * the tree on each device (ptrs_scene_create_device_bvh).  The film of devices[0] is the root. */
int32_t ptrs_multi_create(const PtrsSceneDesc* desc, int32_t n_devices, const int32_t* devices,
                          int32_t device_bvh, PtrsMultiScene** out);
int32_t ptrs_multi_destroy(PtrsMultiScene* multi);
int32_t ptrs_multi_device_count(const PtrsMultiScene* multi, int32_t* n_devices);
/* PathIntegrator::render on all devices: clears the per-device films, renders shard g of the sample
 * numbers selected by `params` on device g, reduces the films into the root film and — if host_rgbw is
 * not NULL — downloads the raw sums (W*H*4 floats, as ptrs_film_download).  per_device_stats (may be
 * NULL) receives n_devices records; total_ms (may be NULL) the wall time of the whole call. */
int32_t ptrs_multi_render(PtrsMultiScene* multi, const PtrsCamera* camera, const PtrsRenderParams* params,
                          float* host_rgbw, PtrsStats* per_device_stats, float* total_ms);
/* the same restricted to a rectangle of sample positions, as ptrs_render_region; the reduce and the download still
 * cover the whole film.  ptrs_multi_render is this call with the whole sample bounds. */
int32_t ptrs_multi_render_region(PtrsMultiScene* multi, const PtrsCamera* camera, const PtrsRenderParams* params,
                                 const int32_t sample_rect[4], float* host_rgbw, PtrsStats* per_device_stats, float* total_ms);
/* the root film (owned by the handle; valid until the next ptrs_multi_render with another resolution) for
 * ptrs_film_resolve / ptrs_film_resolve_srgb8 */
int32_t ptrs_multi_root_film(PtrsMultiScene* multi, PtrsFilm** film);
/* the replica on device index g, e.g. for ptrs_intersect */
int32_t ptrs_multi_scene(PtrsMultiScene* multi, int32_t g, PtrsScene** scene);

/* (b) one process per GPU (MPI / torchrun style): rank 0 obtains an id, ships its 128 bytes to the other
 * ranks by whatever channel the host has, every rank joins on its current device; then each rank renders
 * its shard (PtrsRenderParams.sample_stride / sample_phase) and calls ptrs_film_reduce. */
int32_t ptrs_comm_unique_id(uint8_t id[PTRS_COMM_ID_BYTES]);
int32_t ptrs_comm_init_rank(const uint8_t id[PTRS_COMM_ID_BYTES], int32_t n_ranks, int32_t rank, PtrsComm** out);
int32_t ptrs_comm_destroy(PtrsComm* comm);
int32_t ptrs_comm_info(const PtrsComm* comm, int32_t* n_ranks, int32_t* rank);
/* Film::merge_film_tile across ranks (film.rs:213-228): sum of every rank's film into `root`'s film, in
 * place, enqueued on `stream` (ncclReduce, f32 sum, W*H*4 elements).  Films of the other ranks are unchanged. */
int32_t ptrs_film_reduce(PtrsComm* comm, PtrsFilm* film, int32_t root, void* stream);

/* Parity probes: single stages of the path, for bit-level checks against the oracle. */
/* SobolSampler::{start_pixel, get_index_for_sample, sample_dimension} (sampler/sobol.rs:81-193):
 * out[i * n_dims + k] = sample_dimension(index(pixels[i], sample_nums[i]), dims[k]) */
int32_t ptrs_sobol_samples(const PtrsCamera* camera, const PtrsRenderParams* params,
                           const int32_t* pixels_xy, const int32_t* sample_nums, size_t n,
                           const int32_t* dims, size_t n_dims, float* out, uint64_t* out_index);
/* camera sample + Camera::generate_ray_differential + scale_differentials (mod.rs:59-81,
 * ray.rs:30-35): rays[i], p_film[2i..], rx/ry directions [6i..] */
int32_t ptrs_generate_rays(const PtrsCamera* camera, const PtrsRenderParams* params,
                           const int32_t* pixels_xy, const int32_t* sample_nums, size_t n,
                           PtrsRay* rays, float* p_film, float* rxry_dir);

/* Single BxDFs (bxdf/mod.rs:184-193 and the Fresnel / microfacet types they own), for lobe-by-lobe comparison with
 * the CPU path.  kind / fresnel are the enums below; field use by kind:
 *   r   Lambertian r, SpecularReflection r, FresnelSpecular r, MicrofacetReflection r, FresnelBlend rd, DisneyDiffuse r
 *   t   SpecularTransmission t, FresnelSpecular t, MicrofacetTransmission t, FresnelBlend rs
 *   fa, fb   Fresnel parameters: conductor (eta_t, k) with eta_i = 1; Disney (r0, {metallic, eta, -})
 *   eta_a, eta_b   the dielectric indices of the specular / transmission lobes and of FRESNEL_DIELECTRIC
 *   alpha_x, alpha_y, disney_g   TrowbridgeReitzDistribution (clamped to >= 1e-3 as microfacet.rs:113-116) / the
 *                                separable-G DisneyMicrofacetDistribution (disney.rs:138-170) */
typedef enum PtrsLobeKind {
  PTRS_LOBE_LAMBERTIAN = 0,
  PTRS_LOBE_SPECULAR_REFLECTION = 1,
  PTRS_LOBE_SPECULAR_TRANSMISSION = 2,
  PTRS_LOBE_FRESNEL_SPECULAR = 3,
  PTRS_LOBE_MICROFACET_REFLECTION = 4,
  PTRS_LOBE_MICROFACET_TRANSMISSION = 5,
  PTRS_LOBE_FRESNEL_BLEND = 6,
  PTRS_LOBE_DISNEY_DIFFUSE = 7
} PtrsLobeKind;
typedef enum PtrsFresnelKind {
  PTRS_FRESNEL_DIELECTRIC = 0,
  PTRS_FRESNEL_CONDUCTOR = 1,
  PTRS_FRESNEL_DISNEY = 2,
  PTRS_FRESNEL_NOOP = 3
} PtrsFresnelKind;
typedef struct PtrsLobeDesc {
  int32_t kind;
  int32_t fresnel;
  float r[3];
  float t[3];
  float fa[3];
  float fb[3];
  float eta_a, eta_b;
  float alpha_x, alpha_y;
  int32_t disney_g;
  int32_t pad;
} PtrsLobeDesc;
/* `flags`: PTRS_RENDER_EXACT_SHADING evaluates with the exact units' arithmetic (IEEE division / square root, no FMA
 * contraction), 0 with the default shade kernels' arithmetic.  Directions are in the local shading frame (z = normal).
 * BxDF::f and BxDF::pdf: out[4 i ..] = f.r, f.g, f.b, pdf */
int32_t ptrs_bxdf_eval(const PtrsLobeDesc* lobe, const float* wo /* 3n */, const float* wi /* 3n */, size_t n,
                       int32_t flags, float* out /* 4n */);
/* BxDF::sample_f: out[8 i ..] = wi.x, wi.y, wi.z, f.r, f.g, f.b, pdf, sampled BxDFType bits (as a float) */
int32_t ptrs_bxdf_sample(const PtrsLobeDesc* lobe, const float* wo /* 3n */, const float* u /* 2n */, size_t n,
                         int32_t flags, float* out /* 8n */);
/* Light::sample_li (light.rs) of light `light` from reference points ref_p with normals ref_n (p_error = 0), followed
 * by the visibility segment VisibilityTester / Interaction::spawn_ray_to_it builds (light.rs:33-42, interaction.rs:50-59):
 * out[16 i ..] = Li rgb, wi xyz, pdf, segment origin xyz, segment direction xyz (un-normalised), 3 x pad */
int32_t ptrs_light_sample(PtrsScene* scene, int32_t light, const float* ref_p /* 3n */, const float* ref_n /* 3n */,
                          const float* u /* 2n */, size_t n, int32_t flags, float* out /* 16n */);
/* Light::pdf_li for directions wi from the same kind of reference points */
int32_t ptrs_light_pdf(PtrsScene* scene, int32_t light, const float* ref_p /* 3n */, const float* ref_n /* 3n */,
                       const float* wi /* 3n */, size_t n, int32_t flags, float* out /* n */);

#ifdef __cplusplus
}
#endif
#endif /* PTRS_B200_H */
