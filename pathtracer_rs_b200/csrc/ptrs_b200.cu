// libptrs_b200.so — C ABI (include/ptrs_b200.h) over the sm_100a wavefront path tracer.
// Host side: scene upload and re-layout, film, the per-batch launch schedule, statistics.
// There is deliberately no CPU code path here: without a CUDA device every entry point fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "handles.hpp"
#include "launch.hpp"
#include "wavefront.cuh"

using namespace ptrs;

// Sobol tables (pathtracer_rs_b200/data/sobol_tables.bin) linked into the library by sobol_blob.S
extern "C" const unsigned char ptrs_sobol_blob[];
extern "C" const unsigned char ptrs_sobol_blob_end[];

namespace {

thread_local std::string g_err;
int32_t fail(int32_t code, const std::string& msg) {
  g_err = msg;
  return code;
}
}  // namespace
int32_t ptrs::set_error(int32_t code, const std::string& msg) { return fail(code, msg); }
namespace {
#define CUDA_TRY(expr)                                                                                         \
  do {                                                                                                         \
    cudaError_t e__ = (expr);                                                                                  \
    if (e__ != cudaSuccess) return fail(PTRS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

struct SobolHost {
  uint32_t n_dims = 0, n_cols = 0;
  const uint32_t* matrices = nullptr;
  std::vector<std::vector<uint64_t>> vdc, vdc_inv;
  bool ok = false;
};
const SobolHost& sobol_host() {
  static SobolHost h;
  static std::once_flag once;
  std::call_once(once, [] {
    const unsigned char* p = ptrs_sobol_blob;
    const unsigned char* end = ptrs_sobol_blob_end;
    if (end - p < 20 || std::memcmp(p, "SOBL", 4) != 0) return;
    uint32_t hdr[4];
    std::memcpy(hdr, p + 4, 16);
    p += 20;
    h.n_dims = hdr[0];
    h.n_cols = hdr[1];
    h.matrices = reinterpret_cast<const uint32_t*>(p);
    p += (size_t)hdr[0] * hdr[1] * 4;
    auto rd = [&](std::vector<std::vector<uint64_t>>& dst, uint32_t n) {
      for (uint32_t i = 0; i < n; ++i) {
        uint32_t len;
        std::memcpy(&len, p, 4);
        p += 4;
        std::vector<uint64_t> v(len);
        std::memcpy(v.data(), p, (size_t)len * 8);
        p += (size_t)len * 8;
        dst.push_back(std::move(v));
      }
    };
    rd(h.vdc, hdr[2]);
    rd(h.vdc_inv, hdr[3]);
    h.ok = p <= end && h.n_cols == PT_SOBOL_COLS;
  });
  return h;
}

// Device buffers come from a PRIVATE stream-ordered memory pool per device (cudaMemPoolCreate, release threshold
// raised), so that freeing and re-creating a scene or a multi-GB path workspace re-uses the reservation instead
// of unmapping / mapping it (cudaFree of the 6 GB workspace alone costs ~0.3 s) — without touching the device's
// default pool, which other libraries in the process (PyTorch's cudaMallocAsync backend) share.
// ptrs_trim_memory() hands the cached memory back to the driver.
struct DevicePools {
  std::mutex mu;
  cudaMemPool_t pool[PT_MAX_DEVICES] = {};
};
DevicePools& device_pools() {
  static DevicePools p;
  return p;
}
cudaError_t pool_of_current_device(cudaMemPool_t* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= PT_MAX_DEVICES) return cudaErrorInvalidDevice;
  DevicePools& P = device_pools();
  std::lock_guard<std::mutex> lock(P.mu);
  if (!P.pool[dev]) {
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool;
    e = cudaMemPoolCreate(&pool, &props);
    if (e != cudaSuccess) return e;
    uint64_t keep = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    P.pool[dev] = pool;
  }
  *out = P.pool[dev];
  return cudaSuccess;
}
}  // namespace

namespace ptrs {
// stream-ordered allocation from the library's pool of the current device; freed with cudaFreeAsync
cudaError_t pool_alloc(void** p, size_t bytes, cudaStream_t st) {
  cudaMemPool_t pool;
  cudaError_t e = pool_of_current_device(&pool);
  if (e != cudaSuccess) return e;
  return cudaMallocFromPoolAsync(p, bytes, pool, st);
}
}  // namespace ptrs

namespace {

// Entry points run on the device their handle lives on, whatever the calling thread's current device is, and
// leave the thread's current device as they found it.
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    else if (err == cudaSuccess) prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define ON_DEVICE_OF(handle)                                                                        \
  DeviceGuard guard__((handle)->device);                                                            \
  if (guard__.err != cudaSuccess) return fail(PTRS_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(guard__.err))

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    if (count == 0) return cudaSuccess;
    return ptrs::pool_alloc(reinterpret_cast<void**>(&p), count * sizeof(T), (cudaStream_t)0);
  }
  cudaError_t upload(const T* src, size_t count) {
    cudaError_t e = alloc(count);
    if (e != cudaSuccess || count == 0) return e;
    return cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
  }
  void release() {
    if (p) cudaFreeAsync(p, (cudaStream_t)0);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
};

struct Workspace {
  uint32_t cap = 0, rounds = 0;
  DevBuf<PathSlot> slot;
  DevBuf<float4> L, q_hit;
  DevBuf<NeeRec> nee;
  DevBuf<NeeRes> nee_res;
  DevBuf<int> q_ext[2], q_nee, q_class;
  DevBuf<uint32_t> q_ray;
  DevBuf<RoundCounters> counters;
  DevBuf<GlobalCounters> gcount;
  PathArrays arrays() {
    PathArrays a;
    a.slot = slot.p;
    a.L = L.p;
    a.q_hit = q_hit.p;
    a.nee = nee.p;
    a.nee_res = nee_res.p;
    a.q_ray = q_ray.p;
    return a;
  }
  static constexpr uint64_t kBytesPerSlot = sizeof(PathSlot) + 16 + sizeof(NeeRec) + sizeof(NeeRes) + 4 * 5 + (4 + 16) * PT_N_CLASSES;  // 368
  uint64_t bytes() const { return (uint64_t)cap * kBytesPerSlot + (uint64_t)rounds * sizeof(RoundCounters); }
};

}  // namespace

struct PtrsScene {
  int device = 0;
  DevScene dev{};
  DevBuf<float4> nodes, tri_verts;
  DevBuf<float4> wnodes;  // occlusion tree (dev_accel.cuh trace_occlusion), empty when the scene has none
  bool has_area_light = false;  // closest-hit MIS rays exist only for area lights
  DevBuf<uint4> tri_index;
  DevBuf<float4> tri_shade;
  DevBuf<uint32_t> prim_map;  // device-built BVH: BVH position -> caller's primitive index
  float bvh_build_ms = 0.f;
  uint32_t n_dev_nodes = 0;
  uint32_t bvh_depth = 0;  // largest number of pending stack entries a traversal can need
  DevBuf<float> normal, tangent, uv, texels;
  DevBuf<PtrsMesh> meshes;
  DevBuf<PtrsMaterial> materials;
  DevBuf<PtrsTexture> textures;
  DevBuf<PtrsMipMap> mipmaps;
  DevBuf<PtrsLight> lights;
  DevBuf<int> infinite_lights;
  DevBuf<DevEnv> envs;
  std::vector<DevBuf<float>> env_arrays;
  std::vector<DevBuf<uint32_t>> env_guides;
  DevBuf<uint32_t> sobol, split_tab;
  SobolSplit split_cfg{};      // what split_tab currently holds
  SobolConfig split_for{};    // ... and the sampler configuration it was built for
  DevBuf<uint32_t> ticket;
  DevBuf<GlobalCounters> gcount;
  float world_bound[6] = {0, 0, 0, 0, 0, 0};
  uint64_t scene_bytes = 0;
  uint64_t n_texels = 0;                  // floats in the device texel pool
  uint32_t default_cap = 0;               // wavefront batch size when the caller leaves it to the library (default_paths_per_batch)
  std::vector<PtrsMipMap> host_mipmaps;   // the headers as the device holds them (pyramids completed)
  std::vector<DevEnv> host_envs;          // device pointers of the env tables, for ptrs_scene_download_env
  Workspace ws;
  PtrsStats stats{};
  bool count_visits = false;
  bool has_mat[PTRS_MAT_COUNT] = {false, false, false, false, false, false};
  int sm_count = 148;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  std::vector<cudaEvent_t> stage_events;
  ~PtrsScene() {
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : stage_events) cudaEventDestroy(e);
  }
};

namespace {

int32_t build_render_const(const PtrsCamera* cam, const PtrsRenderParams* rp, RenderConst* rc, std::string* why) {
  const SobolHost& sh = sobol_host();
  if (!sh.ok) {
    *why = "embedded Sobol tables are corrupt";
    return PTRS_ERR_INVALID_ARGUMENT;
  }
  if (cam->width <= 0 || cam->height <= 0 || rp->spp <= 0 || rp->max_depth < 0) {
    *why = "bad camera resolution / spp / max_depth";
    return PTRS_ERR_INVALID_ARGUMENT;
  }
  if (!(rp->filter_radius[0] > 0.f) || !(rp->filter_radius[1] > 0.f) || !(rp->filter_radius[0] < 1024.f) || !(rp->filter_radius[1] < 1024.f)) {
    *why = "filter radius must be positive (and finite)";
    return PTRS_ERR_INVALID_ARGUMENT;
  }
  if (rp->max_depth > 120) {  // 8 Sobol dimensions per bounce must stay below 1024 (sobol.rs:178-183 panics)
    *why = "max_depth > 120 would exceed the 1024 Sobol dimensions";
    return PTRS_ERR_UNSUPPORTED;
  }
  std::memset(rc, 0, sizeof(*rc));
  // Film::get_sample_bounds, film.rs:174-185
  const int sbx0 = (int)std::floor(0.5f - rp->filter_radius[0]), sby0 = (int)std::floor(0.5f - rp->filter_radius[1]);
  const int sbx1 = (int)std::ceil((float)cam->width - 0.5f + rp->filter_radius[0]);
  const int sby1 = (int)std::ceil((float)cam->height - 0.5f + rp->filter_radius[1]);
  // SobolSamplerBuilder::new, sobol.rs:35-62
  int64_t spp = rp->spp;
  {
    int64_t v = spp - 1;
    v |= v >> 1; v |= v >> 2; v |= v >> 4; v |= v >> 8; v |= v >> 16; v |= v >> 32;
    spp = v + 1;
  }
  int32_t ext = std::max(sbx1 - sbx0, sby1 - sby0);
  {
    int32_t v = ext - 1;
    v |= v >> 1; v |= v >> 2; v |= v >> 4; v |= v >> 8; v |= v >> 16;
    ext = v + 1;
  }
  uint32_t m = 0;
  while ((1 << (m + 1)) <= ext) ++m;
  if (m < 1 || m > 25 || (uint64_t)m * 2 + (uint64_t)std::ceil(std::log2((double)spp)) > 52) {
    *why = "resolution / spp outside the Sobol tables' range";
    return PTRS_ERR_UNSUPPORTED;
  }
  SobolConfig& sc = rc->sobol;
  sc.bounds_min[0] = sbx0;
  sc.bounds_min[1] = sby0;
  sc.resolution = ext;
  sc.log2_resolution = m;
  sc.n_vdc = (uint32_t)sh.vdc[m - 1].size();
  sc.n_vdc_inv = (uint32_t)sh.vdc_inv[m - 1].size();
  std::memcpy(sc.vdc, sh.vdc[m - 1].data(), sc.n_vdc * 8);
  std::memcpy(sc.vdc_inv, sh.vdc_inv[m - 1].data(), sc.n_vdc_inv * 8);
  sc.spp = (int32_t)spp;
  rc->cam = *cam;
  std::memcpy(rc->filter_table, rp->filter_table, sizeof(rc->filter_table));
  rc->filter_radius[0] = rp->filter_radius[0];
  rc->filter_radius[1] = rp->filter_radius[1];
  rc->inv_filter_radius[0] = 1.f / rp->filter_radius[0];
  rc->inv_filter_radius[1] = 1.f / rp->filter_radius[1];
  rc->diff_scale = 1.0f / std::sqrt((float)spp);
  rc->max_depth = rp->max_depth;
  rc->rr_threshold = rp->rr_threshold;
  rc->rr_start_depth = rp->rr_start_depth;
  rc->rr_enable = rp->rr_enable;
  rc->sb_min[0] = sbx0;
  rc->sb_min[1] = sby0;
  rc->sb_ext[0] = sbx1 - sbx0;
  rc->sb_ext[1] = sby1 - sby0;
  for (int k = 0; k < 2; ++k) {
    rc->rect_min[k] = rc->sb_min[k];
    rc->rect_ext[k] = rc->sb_ext[k];
  }
  if (sbx0 < -32768 || sby0 < -32768 || sbx1 > 32767 || sby1 > 32767) {  // pixel coordinates travel as two int16 in the path record
    *why = "sample bounds outside the 16-bit pixel range of the path record";
    return PTRS_ERR_UNSUPPORTED;
  }
  const int stride = rp->sample_stride > 0 ? rp->sample_stride : 1;
  const int phase = ((rp->sample_phase % stride) + stride) % stride;
  const int s_lo = std::max(rp->sample_begin, 0);
  const int s_hi = rp->sample_end > 0 ? std::min<int64_t>(rp->sample_end, spp) : (int)spp;
  int first = s_lo + ((phase - s_lo % stride) + stride) % stride;
  rc->s_begin = first;
  rc->s_stride = stride;
  rc->s_phase = phase;
  rc->s_count = first < s_hi ? (s_hi - first + stride - 1) / stride : 0;
  return PTRS_OK;
}

int32_t ensure_workspace(PtrsScene* s, uint32_t cap, uint32_t rounds) {
  Workspace& w = s->ws;
  if (w.cap >= cap && w.rounds >= rounds) return PTRS_OK;
  cap = std::max(cap, w.cap);
  rounds = std::max(rounds, w.rounds);
#define WS_ALLOC(buf, count) \
  if ((buf).alloc(count) != cudaSuccess) return fail(PTRS_ERR_OUT_OF_MEMORY, "workspace allocation failed")
  WS_ALLOC(w.slot, cap);
  WS_ALLOC(w.L, cap);
  WS_ALLOC(w.nee, cap);
  WS_ALLOC(w.nee_res, cap);
  WS_ALLOC(w.q_hit, (size_t)cap * PT_N_CLASSES);
  WS_ALLOC(w.q_ext[0], cap);
  WS_ALLOC(w.q_ext[1], cap);
  WS_ALLOC(w.q_nee, cap);
  WS_ALLOC(w.q_ray, (size_t)cap * 2);
  WS_ALLOC(w.q_class, (size_t)cap * PT_N_CLASSES);
  WS_ALLOC(w.counters, rounds + 1);
  WS_ALLOC(w.gcount, 1);
#undef WS_ALLOC
  if (cudaStreamSynchronize((cudaStream_t)0) != cudaSuccess) return fail(PTRS_ERR_CUDA, "workspace allocation failed");  // allocations are ordered on the legacy stream; the render may use another
  w.cap = cap;
  w.rounds = rounds;
  return PTRS_OK;
}

// Sobol split tables (dev_sobol.cuh): rows = spp sample numbers + x extent + y extent of the sample bounds,
// `stride` dimensions each — enough for every draw of a max_depth path (2 camera dimensions, the 4 -> 5 skip,
// at most 8 per bounce); built on the device by the reference's own index / sample functions and cached
// until the sampler configuration changes.
int32_t plan_split(RenderConst* rc) {
  SobolSplit& sp = rc->split;
  const uint32_t want = 8u + 8u * ((uint32_t)rc->max_depth + 2u);
  sp.stride = std::min<uint32_t>(1024u, (want + 3u) & ~3u);
  sp.row_x = (uint32_t)rc->sobol.spp;
  sp.row_y = sp.row_x + (uint32_t)rc->sb_ext[0];
  sp.n_rows = sp.row_y + (uint32_t)rc->sb_ext[1];
  sp.tab = nullptr;
  if ((uint64_t)sp.n_rows * sp.stride > 0xffffffffull) return PTRS_ERR_UNSUPPORTED;  // element offsets are 32 bit
  return PTRS_OK;
}
int32_t build_split(RenderConst* rc, const uint32_t* d_sobol, DevBuf<uint32_t>* tab, cudaStream_t st) {
  if (tab->alloc((size_t)rc->split.n_rows * rc->split.stride) != cudaSuccess) return fail(PTRS_ERR_OUT_OF_MEMORY, "Sobol split table allocation failed");
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)0));  // the allocation is ordered on the legacy stream
  rc->split.tab = tab->p;
  launch_sobol_split_build(st, *rc, d_sobol, tab->p);
  CUDA_TRY(cudaGetLastError());
  return PTRS_OK;
}
int32_t ensure_split(PtrsScene* s, RenderConst* rc, cudaStream_t st) {
  int32_t r = plan_split(rc);
  if (r != PTRS_OK) return fail(r, "resolution x max_depth too large for the Sobol split tables");
  const SobolSplit& want = rc->split;
  const SobolSplit& have = s->split_cfg;
  if (s->split_tab.p && have.stride >= want.stride && have.row_x == want.row_x && have.row_y == want.row_y && have.n_rows == want.n_rows &&
      std::memcmp(&s->split_for, &rc->sobol, sizeof(SobolConfig)) == 0) {
    rc->split = have;
    return PTRS_OK;
  }
  r = build_split(rc, s->dev.sobol, &s->split_tab, st);
  if (r != PTRS_OK) return r;
  s->split_cfg = rc->split;
  s->split_for = rc->sobol;
  s->stats.launches += 1;
  return PTRS_OK;
}

// (pixel, sample number) lists of the probes: inside the sample bounds and below spp, as in the reference's loops
int32_t check_pixel_list(const RenderConst& rc, const int32_t* xy, const int32_t* sn, size_t n) {
  for (size_t i = 0; i < n; ++i) {
    const int x = xy[2 * i] - rc.sb_min[0], y = xy[2 * i + 1] - rc.sb_min[1];
    if (x < 0 || y < 0 || x >= rc.sb_ext[0] || y >= rc.sb_ext[1] || sn[i] < 0 || sn[i] >= rc.sobol.spp)
      return fail(PTRS_ERR_INVALID_ARGUMENT, "pixel outside the sample bounds or sample number outside [0, spp)");
  }
  return PTRS_OK;
}

enum { ST_GENERATE, ST_EXTEND, ST_SHADE, ST_CONNECT, ST_ACCUMULATE, ST_RESOLVE, ST_COUNT };
struct StageTimer {
  PtrsScene* s;
  cudaStream_t st;
  size_t used = 0;
  std::vector<std::pair<int, size_t>> spans;  // (stage id, first event index)
  cudaEvent_t next() {
    if (used == s->stage_events.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      s->stage_events.push_back(e);
    }
    return s->stage_events[used++];
  }
  void begin(int stage) {
    spans.emplace_back(stage, used);
    cudaEventRecord(next(), st);
  }
  void end() { cudaEventRecord(next(), st); }
  void collect(float ms[ST_COUNT]) {  // call after a stream sync
    for (auto& sp_ : spans) {
      float t = 0.f;
      cudaEventElapsedTime(&t, s->stage_events[sp_.second], s->stage_events[sp_.second + 1]);
      ms[sp_.first] += t;
    }
    spans.clear();
    used = 0;
  }
};

// One wavefront batch: `n_work` path slots already described by (work_base | lists); runs rounds until
// every path has ended.  Leaves per-path radiance in ws.L.
int32_t run_batch(PtrsScene* s, const RenderConst& rc, bool exact_shading, uint64_t work_base, uint32_t n_work, const int* d_list_xy, const int* d_list_s,
                  cudaStream_t st, StageTimer& tm, uint64_t* ext_rays) {
  Workspace& w = s->ws;
  PathArrays P = w.arrays();
  const uint32_t cap = w.cap;
  const int sm = s->sm_count;
  CUDA_TRY(cudaMemsetAsync(w.counters.p, 0, (size_t)(w.rounds + 1) * sizeof(RoundCounters), st));
  tm.begin(ST_GENERATE);
  launch_generate(st, sm, rc, s->dev.sobol, P, work_base, n_work, d_list_xy, d_list_s, w.q_ext[0].p, w.counters.p);
  tm.end();
  s->stats.launches += 1;
  uint32_t round = 0;
  const uint32_t planned = (uint32_t)rc.max_depth + 1;
  std::vector<RoundCounters> host_ctr;
  for (;;) {
    const uint32_t upto = std::min(std::max(planned, round + 4), w.rounds);
    for (; round < upto; ++round) {
      RoundCounters* c = w.counters.p + round;
      int* q_in = w.q_ext[round & 1].p;
      int* q_out = w.q_ext[(round + 1) & 1].p;
      tm.begin(ST_EXTEND);
      launch_extend(st, sm, s->count_visits, s->dev, P, q_in, w.q_class.p, cap, c, w.gcount.p);
      s->stats.extend_launches += 1;
      tm.end();
      tm.begin(ST_SHADE);
      if (s->dev.n_infinite_lights > 0) {
        launch_shade_miss(st, sm, s->dev, P, w.q_class.p + (size_t)PT_CLASS_MISS * cap, c);
        s->stats.launches += 1;
      }
#define SHADE(M)                                                                                                               \
  if (s_has_mat[M]) {                                                                                                          \
    if (exact_shading)                                                                                                         \
      launch_shade_exact_##M(st, sm, rc, s->dev, P, w.q_class.p + (size_t)(M)*cap, w.q_hit.p + (size_t)(M)*cap, q_out, w.q_nee.p, c, c + 1); \
    else                                                                                                                       \
      launch_shade_##M(st, sm, rc, s->dev, P, w.q_class.p + (size_t)(M)*cap, w.q_hit.p + (size_t)(M)*cap, q_out, w.q_nee.p, c, c + 1);       \
    s->stats.launches += 1;                                                                                                    \
  }
      const bool* s_has_mat = s->has_mat;
      SHADE(0) SHADE(1) SHADE(2) SHADE(3) SHADE(4) SHADE(5)
#undef SHADE
      tm.end();
      tm.begin(ST_CONNECT);
      if (s->dev.n_lights > 0) {
        // any-hit rays over the occlusion tree, closest-hit MIS rays (area lights only) over the reference tree; in stats
        // mode everything takes the reference walk, so that the visit counters stay the reference's
        if (!s->count_visits && s->dev.n_wnodes > 0) {
          launch_occlusion(st, sm, s->dev, P, c, w.gcount.p);
          if (s->has_area_light) {
            launch_connect(st, sm, false, s->dev, P, cap, true, c, w.gcount.p);
            s->stats.launches += 1;
          }
        } else {
          launch_connect(st, sm, s->count_visits, s->dev, P, cap, false, c, w.gcount.p);
        }
        tm.end();
        tm.begin(ST_RESOLVE);
        launch_connect_resolve(st, sm, s->dev, P, w.q_nee.p, c);
        s->stats.launches += 1;
        s->stats.connect_launches += 1;
        s->stats.launches += 1;
      }
      tm.end();
      s->stats.launches += 1;
    }
    // all planned rounds are enqueued: read the queue lengths back once (also the ray statistics)
    host_ctr.resize(round + 1);
    CUDA_TRY(cudaMemcpyAsync(host_ctr.data(), w.counters.p, (size_t)(round + 1) * sizeof(RoundCounters), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (host_ctr[round].n_ext == 0 || round >= w.rounds) break;  // only null-BSDF chains need extra rounds
  }
  for (uint32_t r = 0; r < round; ++r) *ext_rays += host_ctr[r].n_ext;
  if (host_ctr[round].n_ext != 0) return fail(PTRS_ERR_UNSUPPORTED, "paths still alive after the maximum number of wavefront rounds");
  return PTRS_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int32_t ptrs_abi_version(void) { return PTRS_ABI_VERSION; }
const char* ptrs_last_error(void) { return g_err.c_str(); }

int32_t ptrs_device_count(int32_t* count) {
  int n = 0;
  CUDA_TRY(cudaGetDeviceCount(&n));
  *count = n;
  return PTRS_OK;
}
int32_t ptrs_set_device(int32_t device) {
  CUDA_TRY(cudaSetDevice(device));
  return PTRS_OK;
}

// The occlusion tree (dev_accel.cuh, trace_occlusion) collapsed from the reference's flattened tree (depth-first preorder,
// first child at i + 1, second at `offset`).  Greedy: a wide node starts from the two children of a reference interior node
// and, while it has fewer than four slots, replaces the interior slot of largest surface area by its two children.  Any
// collapse is exact; this choice only favours speed.  Returns false, and the scene traces its any-hit rays over the
// reference tree, when the tree cannot be collapsed exactly: an interior box that does not contain a child's box (the
// reference builder never makes one), or a leaf the 4-byte child word cannot hold (more than 16 primitives, or primitives
// beyond 2^27).
static bool build_occlusion_tree(const PtrsBvhNode* nodes, uint32_t n_nodes, std::vector<float4>* out) {
  auto contains = [&](const PtrsBvhNode& a, const PtrsBvhNode& b) {
    for (int k = 0; k < 3; ++k)
      if (!(a.bounds_min[k] <= b.bounds_min[k]) || !(a.bounds_max[k] >= b.bounds_max[k])) return false;
    return true;
  };
  for (uint32_t i = 0; i < n_nodes; ++i) {
    const PtrsBvhNode& n = nodes[i];
    if (n.n_prims > 0) {
      if (n.n_prims > 16 || (uint64_t)n.offset + n.n_prims > (1u << 27)) return false;
    } else if (!contains(n, nodes[i + 1]) || !contains(n, nodes[n.offset])) {
      return false;
    }
  }
  auto area = [&](uint32_t i) {
    const PtrsBvhNode& n = nodes[i];
    const float dx = n.bounds_max[0] - n.bounds_min[0], dy = n.bounds_max[1] - n.bounds_min[1], dz = n.bounds_max[2] - n.bounds_min[2];
    return dx * dy + dy * dz + dz * dx;
  };
  out->clear();
  std::vector<std::pair<uint32_t, uint32_t>> todo{{0u, 0u}};  // (reference node, wide node)
  out->resize(8);
  while (!todo.empty()) {
    const auto [r, w] = todo.back();
    todo.pop_back();
    std::vector<uint32_t> slot;
    if (nodes[r].n_prims > 0) slot.push_back(r);  // a single-leaf tree: its root alone
    else slot = {r + 1, nodes[r].offset};
    while (slot.size() < 4) {
      int best = -1;
      for (int k = 0; k < (int)slot.size(); ++k)
        if (nodes[slot[k]].n_prims == 0 && (best < 0 || area(slot[k]) > area(slot[best]))) best = k;
      if (best < 0) break;
      const uint32_t c = slot[best];
      slot[best] = c + 1;
      slot.push_back(nodes[c].offset);
    }
    float lo[3][4], hi[3][4];
    uint32_t child[4];
    for (int k = 0; k < 4; ++k) {
      if (k >= (int)slot.size()) {  // empty slot: an empty box and the word PT_W_NONE
        for (int a = 0; a < 3; ++a) {
          lo[a][k] = INFINITY;
          hi[a][k] = -INFINITY;
        }
        child[k] = PT_W_NONE;
        continue;
      }
      const PtrsBvhNode& n = nodes[slot[k]];
      for (int a = 0; a < 3; ++a) {
        lo[a][k] = n.bounds_min[a];
        hi[a][k] = n.bounds_max[a];
      }
      if (n.n_prims > 0) {
        child[k] = PT_W_LEAF_BIT | ((uint32_t)(n.n_prims - 1) << 27) | n.offset;
      } else {
        child[k] = (uint32_t)(out->size() / 8);
        todo.emplace_back(slot[k], child[k]);
        out->resize(out->size() + 8);
      }
    }
    float4* rec = out->data() + 8 * (size_t)w;
    for (int a = 0; a < 3; ++a) {
      rec[2 * a] = make_float4(lo[a][0], lo[a][1], lo[a][2], lo[a][3]);
      rec[2 * a + 1] = make_float4(hi[a][0], hi[a][1], hi[a][2], hi[a][3]);
    }
    std::memcpy(&rec[6], child, 16);
    rec[7] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  return true;
}

// where a scene's tree comes from: the caller's records (ptrs_scene_create), the library's PLOC build
// (ptrs_scene_create_device_bvh) or the reference's SAH build on the device (ptrs_scene_create_sah_bvh)
enum class TreeSource { kCaller, kPloc, kSah };

static int32_t scene_create_impl(const PtrsSceneDesc* d, TreeSource tree, int32_t max_prims_in_node, PtrsScene** out) {
  if (!d || !out) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  const bool device_bvh = tree != TreeSource::kCaller;
  if (d->abi_version != PTRS_ABI_VERSION) return fail(PTRS_ERR_INVALID_ARGUMENT, "PtrsSceneDesc.abi_version mismatch");
  if (d->n_prims > 0 && ((!device_bvh && !d->nodes) || !d->prim_vertex || !d->prim_mesh || !d->prim_material || !d->prim_area_light || !d->pos || !d->meshes))
    return fail(PTRS_ERR_INVALID_ARGUMENT, "missing geometry arrays");
  const SobolHost& sh = sobol_host();
  if (!sh.ok) return fail(PTRS_ERR_INVALID_ARGUMENT, "embedded Sobol tables are corrupt");
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  std::unique_ptr<PtrsScene> s(new PtrsScene());
  s->device = dev;
  CUDA_TRY(cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, dev));
  // The primitive arrays are validated on the device once they are uploaded (validate_prims_on_device below).  The
  // tree is validated here in one pass: the reference's flattened tree is in depth-first preorder (first child at
  // i + 1, second at `offset`, accelerator.rs:348-357), so walking the records in index order with a stack of the
  // second children still owed must consume every record exactly once — which also rules out shared subtrees and
  // cycles, the only inputs that could keep a traversal kernel from terminating.
  uint32_t n_interior = 0;
  if (!device_bvh && d->n_prims > 0) {
    if (d->n_nodes == 0) return fail(PTRS_ERR_INVALID_ARGUMENT, "missing geometry arrays");
    // The walk also measures the tree's depth: a ray's pending stack holds at most one entry per interior
    // ancestor of the node in hand (whichever child it takes first), and the traversal stack has the reference's
    // 64 entries (accelerator.rs:366).  The reference would panic on an out-of-range index there; a deeper tree
    // is refused here instead of being traversed with dropped subtrees.
    std::vector<std::pair<uint32_t, uint32_t>> owed;  // (second child still owed, its depth)
    bool prev_interior = false;
    uint32_t depth = 0, max_interior_depth = 0;
    for (uint32_t i = 0; i < d->n_nodes; ++i) {
      const PtrsBvhNode& n = d->nodes[i];
      if (i > 0 && !prev_interior) {
        if (owed.empty()) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH (records after the end of the tree)");
        if (owed.back().first != i) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH node (second child must follow the first child's subtree)");
        depth = owed.back().second;
        owed.pop_back();
      }
      if (n.n_prims > 0) {
        if ((uint64_t)n.offset + n.n_prims > d->n_prims) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH node");
        prev_interior = false;
      } else {
        if (n.offset >= d->n_nodes || i + 1 >= d->n_nodes || n.axis > 2) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH node");
        if (n.offset <= i + 1) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH node (second child must follow the first child's subtree)");
        max_interior_depth = std::max(max_interior_depth, depth);
        owed.emplace_back(n.offset, depth + 1);
        depth += 1;
        prev_interior = true;
        ++n_interior;
      }
    }
    if (prev_interior || !owed.empty()) return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed BVH (nodes are shared between subtrees)");
    if (n_interior > 0 && max_interior_depth + 1 > PT_STACK_SIZE)
      return fail(PTRS_ERR_UNSUPPORTED, "BVH deeper than the 64-entry traversal stack (accelerator.rs:366)");
    s->bvh_depth = n_interior > 0 ? max_interior_depth + 1 : 0;
  }
  if ((d->n_materials && !d->materials) || (d->n_textures && !d->textures) || (d->n_mipmaps && !d->mipmaps) || (d->n_texels && !d->texels) ||
      (d->n_lights && !d->lights) || (d->n_infinite_lights && !d->infinite_lights) || (d->n_envs && !d->envs) || (d->n_meshes && !d->meshes))
    return fail(PTRS_ERR_INVALID_ARGUMENT, "a table has a non-zero count and a NULL pointer");
  for (uint32_t i = 0; i < d->n_materials; ++i) {
    const PtrsMaterial& m = d->materials[i];
    if (m.type < 0 || m.type >= PTRS_MAT_COUNT) return fail(PTRS_ERR_UNSUPPORTED, "unknown material type");
    s->has_mat[m.type] = true;
    static const int n_tex[PTRS_MAT_COUNT] = {1, 0, 3, 5, 4, 4};
    for (int k = 0; k < n_tex[m.type]; ++k)
      if (m.tex[k] < 0 || (uint32_t)m.tex[k] >= d->n_textures) return fail(PTRS_ERR_INVALID_ARGUMENT, "material texture id out of range");
    if (m.normal_map >= (int32_t)d->n_textures) return fail(PTRS_ERR_INVALID_ARGUMENT, "normal map id out of range");
  }
  for (uint32_t i = 0; i < d->n_textures; ++i) {
    const PtrsTexture& t = d->textures[i];
    if (t.type < PTRS_TEX_CONSTANT || t.type > PTRS_TEX_IMAGE) return fail(PTRS_ERR_UNSUPPORTED, "unknown texture type");
    if (t.type == PTRS_TEX_IMAGE && (t.mip < 0 || (uint32_t)t.mip >= d->n_mipmaps)) return fail(PTRS_ERR_INVALID_ARGUMENT, "image texture without a MIP pyramid");
  }
  for (uint32_t i = 0; i < d->n_mipmaps; ++i) {  // every texel a lookup can address lies inside the pool
    const PtrsMipMap& m = d->mipmaps[i];
    if (m.n_levels < 1 || m.n_levels > PTRS_MAX_MIP_LEVELS || (m.channels != 1 && m.channels != 3) || m.wrap < PTRS_WRAP_REPEAT || m.wrap > PTRS_WRAP_CLAMP)
      return fail(PTRS_ERR_INVALID_ARGUMENT, "malformed MIP pyramid header");
    for (int l = 0; l < m.n_levels; ++l) {
      if (m.width[l] < 1 || m.height[l] < 1) return fail(PTRS_ERR_INVALID_ARGUMENT, "MIP level with a non-positive size");
      const uint64_t need = (uint64_t)m.width[l] * (uint64_t)m.height[l] * (uint64_t)m.channels;
      if (m.level_offset[l] > d->n_texels || need > d->n_texels - m.level_offset[l]) return fail(PTRS_ERR_INVALID_ARGUMENT, "MIP level outside the texel pool");
    }
  }
  for (uint32_t i = 0; i < d->n_meshes; ++i)
    if (d->meshes[i].alpha_tex >= (int32_t)d->n_textures) return fail(PTRS_ERR_INVALID_ARGUMENT, "alpha texture id out of range");
  for (uint32_t i = 0; i < d->n_infinite_lights; ++i) {
    const int32_t li = d->infinite_lights[i];
    if (li < 0 || (uint32_t)li >= d->n_lights || d->lights[li].type != PTRS_LIGHT_INFINITE) return fail(PTRS_ERR_INVALID_ARGUMENT, "infinite_lights names something that is not an infinite light");
  }
  if (d->n_lights > PT_NEE_LIGHT_MASK) return fail(PTRS_ERR_UNSUPPORTED, "more than 2^29 lights");  // the light id shares a word with flags in the direct-lighting record
  for (uint32_t i = 0; i < d->n_lights; ++i) {
    const PtrsLight& l = d->lights[i];
    if (l.type < 0 || l.type > PTRS_LIGHT_INFINITE) return fail(PTRS_ERR_UNSUPPORTED, "unknown light type");
    if (l.type == PTRS_LIGHT_AREA && (l.prim < 0 || (uint32_t)l.prim >= d->n_prims || l.ke_tex < 0 || (uint32_t)l.ke_tex >= d->n_textures))
      return fail(PTRS_ERR_INVALID_ARGUMENT, "area light references an out-of-range primitive / texture");
    if (l.type == PTRS_LIGHT_INFINITE && (l.env < 0 || (uint32_t)l.env >= d->n_envs)) return fail(PTRS_ERR_INVALID_ARGUMENT, "env id out of range");
  }

  for (uint32_t i = 0; i < d->n_meshes; ++i) {
    const uint32_t f = d->meshes[i].flags;
    if (((f & PTRS_MESH_HAS_NORMAL) && !d->normal) || ((f & PTRS_MESH_HAS_TANGENT) && !d->tangent) || ((f & PTRS_MESH_HAS_UV) && !d->uv))
      return fail(PTRS_ERR_INVALID_ARGUMENT, "mesh flags name an attribute pool that is NULL");
  }
  CUDA_TRY(s->meshes.upload(d->meshes, d->n_meshes));
  CUDA_TRY(s->lights.upload(d->lights, d->n_lights));
  uint32_t n_dev_nodes = 0;
  if (d->n_prims > 0) {
    // the caller's arrays go up as they are; re-layout (triangles as 3 x float4 with metadata in .w, nodes as 64-byte
    // sibling pairs) happens on the device
    DevBuf<uint32_t> pv, inv;
    DevBuf<float> pos;
    DevBuf<int32_t> pm, pmat, pal;
    CUDA_TRY(pv.upload(d->prim_vertex, (size_t)d->n_prims * 3));
    CUDA_TRY(pos.upload(d->pos, (size_t)d->n_verts * 3));
    CUDA_TRY(pm.upload(d->prim_mesh, d->n_prims));
    CUDA_TRY(pmat.upload(d->prim_material, d->n_prims));
    CUDA_TRY(pal.upload(d->prim_area_light, d->n_prims));
    const int bad = validate_prims_on_device(0, d->n_prims, pv.p, pm.p, pmat.p, pal.p, d->n_verts, d->n_meshes, d->n_materials, d->n_lights, s->lights.p);
    if (bad < 0) return fail(PTRS_ERR_CUDA, std::string("primitive validation: ") + cudaGetErrorString((cudaError_t)(-bad)));
    if (bad & 1) return fail(PTRS_ERR_INVALID_ARGUMENT, "primitive references an out-of-range mesh / material / light");
    if (bad & 2) return fail(PTRS_ERR_INVALID_ARGUMENT, "vertex index out of range");
    if (bad & 4) return fail(PTRS_ERR_INVALID_ARGUMENT, "prim_area_light names a light that is not an area light");
    CUDA_TRY(s->tri_verts.alloc((size_t)d->n_prims * 3));
    CUDA_TRY(s->tri_index.alloc(d->n_prims));
    if (tree == TreeSource::kPloc) {
      // unordered primitives in, BVH built and triangles laid out on the device (k_bvh.cu)
      CUDA_TRY(inv.alloc(d->n_prims));
      cudaEvent_t e0, e1;
      CUDA_TRY(cudaEventCreate(&e0));
      CUDA_TRY(cudaEventCreate(&e1));
      CUDA_TRY(cudaEventRecord(e0, 0));
      float4* nodes = nullptr;
      uint32_t* perm = nullptr;
      uint32_t dev_depth = 0;
      const int be = build_bvh_on_device(0, d->n_prims, pv.p, pos.p, &nodes, &n_dev_nodes, &perm, &dev_depth);
      if (be != (int)cudaSuccess) return fail(PTRS_ERR_CUDA, std::string("device BVH build: ") + cudaGetErrorString((cudaError_t)be));
      s->nodes.p = nodes;
      s->nodes.n = (size_t)n_dev_nodes * 2;
      s->prim_map.p = perm;
      s->prim_map.n = d->n_prims;
      s->bvh_depth = dev_depth;
      // a radix tree over clustered / coincident centroids can be deeper than the traversal stack (63 Morton bits +
      // the index tie-break); the host-side SAH build (ptrs_scene_create) is the way out for such input
      if (dev_depth > PT_STACK_SIZE) return fail(PTRS_ERR_UNSUPPORTED, "device-built BVH deeper than the 64-entry traversal stack; build the tree on the host");
      launch_assemble_tris(0, d->n_prims, perm, pv.p, pos.p, pm.p, pmat.p, pal.p, s->meshes.p, s->tri_verts.p, s->tri_index.p, inv.p);
      launch_remap_light_prims(0, s->lights.p, d->n_lights, inv.p);
      CUDA_TRY(cudaEventRecord(e1, 0));
      CUDA_TRY(cudaEventSynchronize(e1));
      CUDA_TRY(cudaGetLastError());
      cudaEventElapsedTime(&s->bvh_build_ms, e0, e1);
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      s->scene_bytes += (uint64_t)n_dev_nodes * 32 + (uint64_t)d->n_prims * 4;
      if (n_dev_nodes > 0) {
        float root[8];
        CUDA_TRY(cudaMemcpy(root, s->nodes.p, 32, cudaMemcpyDeviceToHost));
        s->world_bound[0] = root[0];
        s->world_bound[1] = root[1];
        s->world_bound[2] = root[2];
        s->world_bound[3] = root[3];
        s->world_bound[4] = root[4];
        s->world_bound[5] = root[5];
      }
    } else if (tree == TreeSource::kSah) {
      // the reference's tree over the caller's primitive order, built on the device (k_sah.cu); from its records on the
      // scene is assembled as ptrs_scene_create assembles the same records
      CUDA_TRY(inv.alloc(d->n_prims));
      cudaEvent_t e0, e1;
      CUDA_TRY(cudaEventCreate(&e0));
      CUDA_TRY(cudaEventCreate(&e1));
      CUDA_TRY(cudaEventRecord(e0, 0));
      DevBuf<float4> raw;
      uint32_t n_raw = 0, max_depth = 0, *perm = nullptr;
      const int be = build_sah_bvh_on_device(0, d->n_prims, pv.p, pos.p, max_prims_in_node, PT_STACK_SIZE + 1, &raw.p, &n_raw, &perm, &max_depth);
      if (be != (int)cudaSuccess) return fail(PTRS_ERR_CUDA, std::string("device SAH build: ") + cudaGetErrorString((cudaError_t)be));
      raw.n = (size_t)n_raw * 2;
      s->prim_map.p = perm;
      s->prim_map.n = d->n_prims;
      // the depth rule of the caller's trees above: the builder's max_depth counts the deepest leaf, a traversal's stack holds
      // one entry per interior level
      if (max_depth > PT_STACK_SIZE + 1) return fail(PTRS_ERR_UNSUPPORTED, "BVH deeper than the 64-entry traversal stack (accelerator.rs:366)");
      s->bvh_depth = max_depth - 1;
      float4* nodes = nullptr;
      const int pe = pair_layout_on_device(0, raw.p, n_raw, (n_raw - 1) / 2, &nodes, &n_dev_nodes);
      if (pe != (int)cudaSuccess) return fail(PTRS_ERR_CUDA, std::string("BVH re-layout: ") + cudaGetErrorString((cudaError_t)pe));
      s->nodes.p = nodes;
      s->nodes.n = (size_t)n_dev_nodes * 2;
      launch_assemble_tris(0, d->n_prims, perm, pv.p, pos.p, pm.p, pmat.p, pal.p, s->meshes.p, s->tri_verts.p, s->tri_index.p, inv.p);
      launch_remap_light_prims(0, s->lights.p, d->n_lights, inv.p);
      CUDA_TRY(cudaEventRecord(e1, 0));
      CUDA_TRY(cudaEventSynchronize(e1));
      CUDA_TRY(cudaGetLastError());
      cudaEventElapsedTime(&s->bvh_build_ms, e0, e1);
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      s->scene_bytes += (uint64_t)n_dev_nodes * 32 + (uint64_t)d->n_prims * 4;
      // the occlusion tree: the host collapse of ptrs_scene_create, over the records copied back
      const auto t0 = std::chrono::steady_clock::now();
      std::vector<PtrsBvhNode> recs(n_raw);
      CUDA_TRY(cudaMemcpyAsync(recs.data(), raw.p, (size_t)n_raw * 32, cudaMemcpyDeviceToHost, 0));
      CUDA_TRY(cudaStreamSynchronize(0));
      std::memcpy(s->world_bound, recs[0].bounds_min, 12);
      std::memcpy(s->world_bound + 3, recs[0].bounds_max, 12);
      std::vector<float4> wide;
      if (build_occlusion_tree(recs.data(), n_raw, &wide)) {
        CUDA_TRY(s->wnodes.upload(wide.data(), wide.size()));
        s->scene_bytes += (uint64_t)wide.size() * 16;
      }
      if (std::getenv("PTRS_BVH_DEBUG"))
        std::fprintf(stderr, "sah build: occlusion tree (copy-back + host collapse) %9.3f ms\n",
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
      CUDA_TRY(cudaStreamSynchronize(0));  // the staging buffers above are released when this scope ends
    } else {
      // reference-built tree: the 32 B records are kept, but the two children of every interior node are placed side
      // by side (64 B pairs in depth-first order, root alone in slot 0) so that one traversal step reads one
      // contiguous 64 B block; boxes, split axes, leaf ranges and the visit order stay those of the reference
      static_assert(sizeof(PtrsBvhNode) == 32, "LinearBVHNode is 32 bytes");
      DevBuf<float4> raw;
      CUDA_TRY(raw.upload(reinterpret_cast<const float4*>(d->nodes), (size_t)d->n_nodes * 2));
      float4* nodes = nullptr;
      const int pe = pair_layout_on_device(0, raw.p, d->n_nodes, n_interior, &nodes, &n_dev_nodes);
      if (pe != (int)cudaSuccess) return fail(PTRS_ERR_CUDA, std::string("BVH re-layout: ") + cudaGetErrorString((cudaError_t)pe));
      s->nodes.p = nodes;
      s->nodes.n = (size_t)n_dev_nodes * 2;
      s->scene_bytes += (uint64_t)n_dev_nodes * 32;
      // device-built scenes keep the reference walk for any-hit rays: their tree is not the reference's, and the
      // collapse works on the caller's records here on the host
      std::vector<float4> wide;
      if (build_occlusion_tree(d->nodes, d->n_nodes, &wide)) {
        CUDA_TRY(s->wnodes.upload(wide.data(), wide.size()));
        s->scene_bytes += (uint64_t)wide.size() * 16;
      }
      launch_assemble_tris(0, d->n_prims, nullptr, pv.p, pos.p, pm.p, pmat.p, pal.p, s->meshes.p, s->tri_verts.p, s->tri_index.p, nullptr);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaStreamSynchronize(0));  // the staging buffers above are released when this scope ends
    }
  }
  if (n_dev_nodes > (1u << 30)) return fail(PTRS_ERR_UNSUPPORTED, "more than 2^30 BVH nodes");  // packed stack entries, dev_accel.cuh
  if (d->normal) CUDA_TRY(s->normal.upload(d->normal, (size_t)d->n_verts * 3));
  if (d->tangent) CUDA_TRY(s->tangent.upload(d->tangent, (size_t)d->n_verts * 3));
  if (d->uv) CUDA_TRY(s->uv.upload(d->uv, (size_t)d->n_verts * 2));
  CUDA_TRY(s->tri_shade.alloc((size_t)d->n_prims * 4));
  launch_pack_shading(0, d->n_prims, s->tri_verts.p, s->tri_index.p, s->normal.p, s->uv.p, s->tri_shade.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(s->materials.upload(d->materials, d->n_materials));
  CUDA_TRY(s->textures.upload(d->textures, d->n_textures));
  {
    // MIP pyramids.  A PtrsMipMap that carries level 0 only (n_levels == 1 for an image larger than one texel) gets the
    // rest of its pyramid built here, on the device (k_tables.cu; MIPMap::new, texture.rs:345-405).
    std::vector<PtrsMipMap> mips(d->mipmaps, d->mipmaps + d->n_mipmaps);
    std::vector<int> have(d->n_mipmaps, 0);
    bool build_any = false;
    uint64_t total = 0;
    for (uint32_t i = 0; i < d->n_mipmaps; ++i) {
      PtrsMipMap& m = mips[i];
      have[i] = m.n_levels;
      int want = 1;
      for (int e = std::max(m.width[0], m.height[0]); e > 1; e >>= 1) ++want;  // 1 + log2_int(max extent), texture.rs:345
      if (m.n_levels == 1 && want > 1) {
        if ((m.width[0] & (m.width[0] - 1)) || (m.height[0] & (m.height[0] - 1)))
          return fail(PTRS_ERR_UNSUPPORTED, "level 0 of a pyramid to be completed on the device must be a power of two in both axes (the Lanczos resample of MIPMap::new stays with the host)");
        if (want > PTRS_MAX_MIP_LEVELS) return fail(PTRS_ERR_INVALID_ARGUMENT, "MIP pyramid too deep");
        build_any = true;
        m.n_levels = want;
        for (int l = 1; l < want; ++l) {
          m.width[l] = std::max(1, m.width[l - 1] / 2);
          m.height[l] = std::max(1, m.height[l - 1] / 2);
        }
      }
      for (int l = 0; l < m.n_levels; ++l) total += (uint64_t)m.width[l] * m.height[l] * m.channels;
    }
    if (!build_any) {
      CUDA_TRY(s->mipmaps.upload(d->mipmaps, d->n_mipmaps));
      CUDA_TRY(s->texels.upload(d->texels, d->n_texels));
    } else {
      DevBuf<float> in_pool;
      CUDA_TRY(in_pool.upload(d->texels, d->n_texels));
      CUDA_TRY(s->texels.alloc(total));
      uint64_t at = 0;
      for (uint32_t i = 0; i < d->n_mipmaps; ++i) {
        PtrsMipMap& m = mips[i];
        for (int l = 0; l < m.n_levels; ++l) {
          const uint64_t n = (uint64_t)m.width[l] * m.height[l] * m.channels;
          if (l < have[i]) CUDA_TRY(cudaMemcpyAsync(s->texels.p + at, in_pool.p + d->mipmaps[i].level_offset[l], n * 4, cudaMemcpyDeviceToDevice, 0));
          else launch_mip_level(0, s->texels.p + m.level_offset[l - 1], m.width[l - 1], m.height[l - 1], m.channels, m.wrap, s->texels.p + at, m.width[l], m.height[l]);
          m.level_offset[l] = at;
          at += n;
        }
      }
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(s->mipmaps.upload(mips.data(), mips.size()));
      CUDA_TRY(cudaStreamSynchronize(0));  // in_pool is released when this scope ends
    }
    s->n_texels = build_any ? total : d->n_texels;
    s->host_mipmaps = mips;
  }
  CUDA_TRY(s->infinite_lights.upload(d->infinite_lights, d->n_infinite_lights));
  {
    std::vector<DevEnv> envs(d->n_envs);
    s->env_arrays.resize((size_t)d->n_envs * 5);
    s->env_guides.resize((size_t)d->n_envs * 2);
    for (uint32_t i = 0; i < d->n_envs; ++i) {
      PtrsEnvLight e = d->envs[i];
      if (e.mip < 0 || (uint32_t)e.mip >= d->n_mipmaps) return fail(PTRS_ERR_INVALID_ARGUMENT, "incomplete env light");
      const bool build_dist = !e.cond_func && !e.cond_cdf && !e.cond_func_int && !e.marg_func && !e.marg_cdf;
      if (build_dist && (e.nu <= 0 || e.nv <= 0)) {  // light.rs:375-376: twice the map's resolution
        e.nu = 2 * s->host_mipmaps[e.mip].width[0];
        e.nv = 2 * s->host_mipmaps[e.mip].height[0];
      }
      if (e.nu <= 0 || e.nv <= 0 || (!build_dist && (!e.cond_func || !e.cond_cdf || !e.cond_func_int || !e.marg_func || !e.marg_cdf)))
        return fail(PTRS_ERR_INVALID_ARGUMENT, "incomplete env light");
      if ((uint64_t)e.nu * (uint64_t)e.nv > 0x7fffffffull) return fail(PTRS_ERR_UNSUPPORTED, "env distribution too large");
      DevEnv& o = envs[i];
      std::memcpy(o.light_to_world, e.light_to_world, 64);
      std::memcpy(o.world_to_light, e.world_to_light, 64);
      o.mip = e.mip;
      o.nu = e.nu;
      o.nv = e.nv;
      o.marg_func_int = e.marg_func_int;
      DevBuf<float>* a = &s->env_arrays[(size_t)i * 5];
      if (!build_dist) {
        CUDA_TRY(a[0].upload(e.cond_func, (size_t)e.nu * e.nv));
        CUDA_TRY(a[1].upload(e.cond_cdf, (size_t)(e.nu + 1) * e.nv));
        CUDA_TRY(a[2].upload(e.cond_func_int, e.nv));
        CUDA_TRY(a[3].upload(e.marg_func, e.nv));
        CUDA_TRY(a[4].upload(e.marg_cdf, (size_t)e.nv + 1));
      } else {
        // InfiniteAreaLight::new's density and Distribution2D::new on the device (k_tables.cu).  The two libm values of
        // the host path are evaluated here, by the same glibc: sin(pi v') per row and log2 of the filter width.
        if (s->host_mipmaps[e.mip].channels != 3) return fail(PTRS_ERR_INVALID_ARGUMENT, "environment map must be a Spectrum MIPMap");
        CUDA_TRY(a[0].alloc((size_t)e.nu * e.nv));
        CUDA_TRY(a[1].alloc((size_t)(e.nu + 1) * e.nv));
        CUDA_TRY(a[2].alloc(e.nv));
        CUDA_TRY(a[4].alloc((size_t)e.nv + 1));
        std::vector<float> row_sin((size_t)e.nv);
        for (int vv = 0; vv < e.nv; ++vv) {
          const float vp = ((float)vv + 0.5f) / (float)e.nv;
          row_sin[vv] = std::sin(3.14159265358979323846f * vp);
        }
        DevBuf<float> d_sin, d_int;
        CUDA_TRY(d_sin.upload(row_sin.data(), row_sin.size()));
        CUDA_TRY(d_int.alloc(1));
        const float f_width = 0.5f / (float)std::min(e.nu, e.nv);
        const int n_lv = s->host_mipmaps[e.mip].n_levels;
        const float level = (float)n_lv - 1.0f + std::log2(std::fmax(f_width, 1e-8f));  // texture.rs:448-449
        int mode = 2, il = 0;
        float delta = 0.f;
        if (level < 0.0f) mode = 0;
        else if (level >= (float)(n_lv - 1)) mode = 1;
        else {
          const float fl = std::floor(level);
          il = (int)fl;
          delta = level - fl;
        }
        DevScene tmp{};
        tmp.texels = s->texels.p;
        tmp.mipmaps = s->mipmaps.p;
        launch_env_density(0, tmp, e.mip, e.nu, e.nv, d_sin.p, mode, il, delta, a[0].p);
        launch_row_cdf(0, a[0].p, e.nu, e.nv, a[1].p, a[2].p);
        launch_row_cdf(0, a[2].p, e.nv, 1, a[4].p, d_int.p);  // marginal: Distribution1D over the row integrals
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpy(&o.marg_func_int, d_int.p, 4, cudaMemcpyDeviceToHost));
        // marg_func is the row-integral array itself (sampling.rs:196-203): a second device copy keeps ownership simple
        CUDA_TRY(a[3].alloc(e.nv));
        CUDA_TRY(cudaMemcpy(a[3].p, a[2].p, (size_t)e.nv * 4, cudaMemcpyDeviceToDevice));
      }
      o.cond_func = a[0].p;
      o.cond_cdf = a[1].p;
      o.cond_func_int = a[2].p;
      o.marg_func = a[3].p;
      o.marg_cdf = a[4].p;
      auto pow2_ge = [](uint32_t n) {
        uint32_t k = 1;
        while (k < n) k <<= 1;
        return k;
      };
      o.ku = pow2_ge((uint32_t)e.nu);
      o.kv = pow2_ge((uint32_t)e.nv);
      DevBuf<uint32_t>* g = &s->env_guides[(size_t)i * 2];
      CUDA_TRY(g[0].alloc((size_t)e.nv * (o.ku + 1)));
      CUDA_TRY(g[1].alloc((size_t)o.kv + 1));
      launch_build_guide(0, a[1].p, (uint32_t)e.nu + 1, (uint32_t)e.nv, o.ku, g[0].p);
      launch_build_guide(0, a[4].p, (uint32_t)e.nv + 1, 1u, o.kv, g[1].p);
      o.cond_guide = g[0].p;
      o.marg_guide = g[1].p;
      s->scene_bytes += ((size_t)e.nv * (o.ku + 1) + o.kv + 1) * 4;
      s->scene_bytes += ((size_t)e.nu * e.nv * 2 + e.nv * 4 + 1) * 4;
    }
    CUDA_TRY(s->envs.upload(envs.data(), envs.size()));
    s->host_envs = envs;
    if (d->n_envs > 0) CUDA_TRY(cudaDeviceSynchronize());  // guide tables built
  }
  CUDA_TRY(s->sobol.upload(sh.matrices, (size_t)sh.n_dims * sh.n_cols));
  CUDA_TRY(s->ticket.alloc(4));
  CUDA_TRY(s->gcount.alloc(1));
  DevScene& v = s->dev;
  v.nodes = s->nodes.p;
  v.tri_verts = s->tri_verts.p;
  v.tri_index = s->tri_index.p;
  v.tri_shade = s->tri_shade.p;
  v.normal = s->normal.p;
  v.tangent = s->tangent.p;
  v.uv = s->uv.p;
  v.meshes = s->meshes.p;
  v.materials = s->materials.p;
  v.textures = s->textures.p;
  v.mipmaps = s->mipmaps.p;
  v.texels = s->texels.p;
  v.lights = s->lights.p;
  v.infinite_lights = s->infinite_lights.p;
  v.envs = s->envs.p;
  v.sobol = s->sobol.p;
  v.n_nodes = d->n_prims > 0 ? n_dev_nodes : 0u;
  s->n_dev_nodes = v.n_nodes;
  v.n_prims = d->n_prims;
  v.n_lights = d->n_lights;
  v.n_infinite_lights = d->n_infinite_lights;
  v.box_min = n_dev_nodes <= 4096u ? 12u : 20u;
  v.pop_twice = n_dev_nodes > 4096u ? 1u : 0u;
  if (const char* e = std::getenv("PTRS_POP_TWICE")) v.pop_twice = std::atoi(e) != 0;  // tuning only
  // a reference-built tree is walked in the reference's order (dir_is_neg[axis]); a tree built here front to back
  v.dist_order = tree == TreeSource::kPloc ? 1u : 0u;
  if (const char* e = std::getenv("PTRS_DIST_ORDER")) v.dist_order = tree == TreeSource::kPloc && std::atoi(e) != 0;  // tuning only
  if (const char* e = std::getenv("PTRS_BOX_MIN")) v.box_min = (uint32_t)std::max(1, std::min(32, std::atoi(e)));  // tuning only
  v.wnodes = s->wnodes.p;
  v.n_wnodes = d->n_prims > 0 ? (uint32_t)(s->wnodes.n / 8) : 0u;
  for (uint32_t i = 0; i < d->n_lights; ++i) s->has_area_light |= d->lights[i].type == PTRS_LIGHT_AREA;
  v.uses_differentials = 0;
  for (uint32_t i = 0; i < d->n_materials; ++i) {
    static const int n_tex[PTRS_MAT_COUNT] = {1, 0, 3, 5, 4, 4};
    const PtrsMaterial& m = d->materials[i];
    for (int k = 0; k < n_tex[m.type]; ++k) v.uses_differentials |= d->textures[m.tex[k]].type == PTRS_TEX_IMAGE;
    if (m.normal_map >= 0) v.uses_differentials |= d->textures[m.normal_map].type == PTRS_TEX_IMAGE;
  }
  for (uint32_t i = 0; i < d->n_lights; ++i)  // emitted radiance at a camera-ray hit is looked up with the hit's differentials
    if (d->lights[i].type == PTRS_LIGHT_AREA) v.uses_differentials |= d->textures[d->lights[i].ke_tex].type == PTRS_TEX_IMAGE;
  if (!device_bvh && d->n_nodes > 0) {
    std::memcpy(s->world_bound, d->nodes[0].bounds_min, 12);
    std::memcpy(s->world_bound + 3, d->nodes[0].bounds_max, 12);
  }
  s->scene_bytes += (uint64_t)d->n_prims * 128 + (uint64_t)d->n_verts * 4 * ((d->normal ? 3 : 0) + (d->tangent ? 3 : 0) + (d->uv ? 2 : 0)) +
                    s->n_texels * 4 + (uint64_t)sh.n_dims * sh.n_cols * 4;
  CUDA_TRY(cudaEventCreate(&s->ev[0]));
  CUDA_TRY(cudaEventCreate(&s->ev[1]));
  CUDA_TRY(cudaDeviceSynchronize());
  *out = s.release();
  return PTRS_OK;
}

int32_t ptrs_scene_create(const PtrsSceneDesc* d, PtrsScene** out) { return scene_create_impl(d, TreeSource::kCaller, 0, out); }
int32_t ptrs_scene_create_device_bvh(const PtrsSceneDesc* d, PtrsScene** out) { return scene_create_impl(d, TreeSource::kPloc, 0, out); }
int32_t ptrs_scene_create_sah_bvh(const PtrsSceneDesc* d, int32_t max_prims_in_node, PtrsScene** out) {
  // LinearBVHNode counts a leaf's primitives in 16 bits (accelerator.rs:89-95)
  if (max_prims_in_node < 1 || max_prims_in_node > 65535) return fail(PTRS_ERR_INVALID_ARGUMENT, "max_prims_in_node must be in 1..65535");
  return scene_create_impl(d, TreeSource::kSah, max_prims_in_node, out);
}

int32_t ptrs_scene_bvh_info(const PtrsScene* scene, uint32_t* n_nodes, float* device_build_ms) {
  if (!scene) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n_nodes) *n_nodes = scene->n_dev_nodes;
  if (device_build_ms) *device_build_ms = scene->bvh_build_ms;
  return PTRS_OK;
}
int32_t ptrs_scene_download_nodes(const PtrsScene* scene, PtrsBvhNode* nodes, uint32_t capacity, uint32_t* prim_order) {
  if (!scene || !nodes) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (capacity < scene->n_dev_nodes) return fail(PTRS_ERR_INVALID_ARGUMENT, "node capacity too small");
  ON_DEVICE_OF(scene);
  CUDA_TRY(cudaMemcpy(nodes, scene->nodes.p, (size_t)scene->n_dev_nodes * 32, cudaMemcpyDeviceToHost));
  if (prim_order) {
    if (!scene->prim_map.p) return fail(PTRS_ERR_INVALID_ARGUMENT, "the scene keeps the caller's primitive order (host-built BVH)");
    CUDA_TRY(cudaMemcpy(prim_order, scene->prim_map.p, scene->prim_map.n * 4, cudaMemcpyDeviceToHost));
  }
  return PTRS_OK;
}

int32_t ptrs_scene_download_mipmaps(const PtrsScene* scene, PtrsMipMap* mipmaps, uint32_t capacity, uint64_t* n_texels, float* texels, uint64_t texel_capacity) {
  if (!scene) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  ON_DEVICE_OF(scene);
  if (n_texels) *n_texels = scene->n_texels;
  if (mipmaps) {
    if (capacity < scene->host_mipmaps.size()) return fail(PTRS_ERR_INVALID_ARGUMENT, "mipmap capacity too small");
    std::memcpy(mipmaps, scene->host_mipmaps.data(), scene->host_mipmaps.size() * sizeof(PtrsMipMap));
  }
  if (texels) {
    if (texel_capacity < scene->n_texels) return fail(PTRS_ERR_INVALID_ARGUMENT, "texel capacity too small");
    CUDA_TRY(cudaMemcpy(texels, scene->texels.p, scene->n_texels * 4, cudaMemcpyDeviceToHost));
  }
  return PTRS_OK;
}

int32_t ptrs_scene_download_env(const PtrsScene* scene, int32_t env, int32_t* nu, int32_t* nv, float* cond_func, float* cond_cdf, float* cond_func_int,
                                float* marg_cdf, float* marg_func_int) {
  if (!scene || env < 0 || (size_t)env >= scene->host_envs.size()) return fail(PTRS_ERR_INVALID_ARGUMENT, "env index out of range");
  ON_DEVICE_OF(scene);
  const DevEnv& e = scene->host_envs[env];
  if (nu) *nu = e.nu;
  if (nv) *nv = e.nv;
  if (cond_func) CUDA_TRY(cudaMemcpy(cond_func, e.cond_func, (size_t)e.nu * e.nv * 4, cudaMemcpyDeviceToHost));
  if (cond_cdf) CUDA_TRY(cudaMemcpy(cond_cdf, e.cond_cdf, (size_t)(e.nu + 1) * e.nv * 4, cudaMemcpyDeviceToHost));
  if (cond_func_int) CUDA_TRY(cudaMemcpy(cond_func_int, e.cond_func_int, (size_t)e.nv * 4, cudaMemcpyDeviceToHost));
  if (marg_cdf) CUDA_TRY(cudaMemcpy(marg_cdf, e.marg_cdf, ((size_t)e.nv + 1) * 4, cudaMemcpyDeviceToHost));
  if (marg_func_int) *marg_func_int = e.marg_func_int;
  return PTRS_OK;
}

int32_t ptrs_scene_destroy(PtrsScene* scene) {
  if (!scene) return PTRS_OK;
  ON_DEVICE_OF(scene);
  cudaDeviceSynchronize();
  delete scene;
  return PTRS_OK;
}

int32_t ptrs_trim_memory(void) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceSynchronize());
  ptrs::release_bvh_build_cache();
  CUDA_TRY(cudaDeviceSynchronize());
  cudaMemPool_t pool;
  CUDA_TRY(pool_of_current_device(&pool));
  CUDA_TRY(cudaMemPoolTrimTo(pool, 0));
  return PTRS_OK;
}

static int32_t read_bandwidth_impl(size_t bytes, int32_t reps, bool gather, float* gb_per_s) {
  if (!gb_per_s || bytes < 64 || reps < 1) return fail(PTRS_ERR_INVALID_ARGUMENT, "bad argument");
  int dev = 0, sm = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev));
  DevBuf<float4> buf;
  DevBuf<uint32_t> sink;
  const size_t n_pairs = bytes / 32;
  CUDA_TRY(buf.alloc(n_pairs * 2));
  CUDA_TRY(sink.alloc(1));
  CUDA_TRY(cudaMemsetAsync(buf.p, 0, n_pairs * 32, 0));
  uint64_t n_gathers = 0;
  if (gather) launch_gather_probe(0, sm, buf.p, n_pairs / 2, reps, sink.p, &n_gathers);
  launch_read_probe(0, sm, buf.p, n_pairs, 2, sink.p);  // warm-up: code, TLB, and (for a small buffer) the L2 fill
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  CUDA_TRY(cudaEventRecord(e0, 0));
  if (gather) launch_gather_probe(0, sm, buf.p, n_pairs / 2, reps, sink.p, &n_gathers);
  else launch_read_probe(0, sm, buf.p, n_pairs, reps, sink.p);
  CUDA_TRY(cudaEventRecord(e1, 0));
  CUDA_TRY(cudaEventSynchronize(e1));
  CUDA_TRY(cudaGetLastError());
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *gb_per_s = gather ? (float)((double)n_gathers * 64.0 / (ms * 1e-3) / 1e9) : (float)((double)n_pairs * 32.0 * reps / (ms * 1e-3) / 1e9);
  return PTRS_OK;
}

int32_t ptrs_read_bandwidth(size_t bytes, int32_t reps, float* gb_per_s) { return read_bandwidth_impl(bytes, reps, false, gb_per_s); }
int32_t ptrs_gather_bandwidth(size_t bytes, int32_t gathers_per_thread, float* gb_per_s) { return read_bandwidth_impl(bytes, gathers_per_thread, true, gb_per_s); }

int32_t ptrs_scene_world_bound(const PtrsScene* scene, float out[6]) {
  if (!scene || !out) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  std::memcpy(out, scene->world_bound, 24);
  return PTRS_OK;
}
uint64_t ptrs_scene_device_bytes(const PtrsScene* scene) { return scene ? scene->scene_bytes + scene->ws.bytes() : 0; }

// ---- intersect -----------------------------------------------------------------------------------
static int32_t do_intersect(PtrsScene* s, const PtrsRay* d_rays, size_t n, PtrsHit* d_hits, uint8_t* d_occ, bool any_hit, bool count,
                                cudaStream_t st) {
  if (n > 0xfffffff0ull) return fail(PTRS_ERR_INVALID_ARGUMENT, "too many rays in one call");
  ON_DEVICE_OF(s);
  CUDA_TRY(cudaMemsetAsync(s->ticket.p, 0, 16, st));
  if (count) CUDA_TRY(cudaMemsetAsync(s->gcount.p, 0, sizeof(GlobalCounters), st));
  launch_intersect(st, s->sm_count, any_hit, count, s->dev, d_rays, (uint32_t)n, d_hits, d_occ, s->ticket.p, s->gcount.p, s->prim_map.p);
  CUDA_TRY(cudaGetLastError());
  return PTRS_OK;
}

int32_t ptrs_intersect_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n, PtrsHit* d_hits, void* stream) {
  if (!scene || (n && (!d_rays || !d_hits))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  return do_intersect(scene, d_rays, n, d_hits, nullptr, false, false, (cudaStream_t)stream);
}
int32_t ptrs_intersect_p_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n, uint8_t* d_occ, void* stream) {
  if (!scene || (n && (!d_rays || !d_occ))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  return do_intersect(scene, d_rays, n, nullptr, d_occ, true, false, (cudaStream_t)stream);
}
int32_t ptrs_intersect_counted_device(PtrsScene* scene, const PtrsRay* d_rays, size_t n, PtrsHit* d_hits, int32_t any_hit, uint8_t* d_occ,
                                      uint64_t* nodes_tested, uint64_t* tris_tested, void* stream) {
  if (!scene || (n && !d_rays) || (n && (any_hit ? !d_occ : !d_hits))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  GlobalCounters g{};
  ON_DEVICE_OF(scene);
  if (n) {
    int32_t rc = do_intersect(scene, d_rays, n, d_hits, d_occ, any_hit != 0, true, (cudaStream_t)stream);
    if (rc != PTRS_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(&g, scene->gcount.p, sizeof(g), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  }
  if (nodes_tested) *nodes_tested = g.nodes_tested;
  if (tris_tested) *tris_tested = g.tris_tested;
  return PTRS_OK;
}

int32_t ptrs_intersect(PtrsScene* scene, const PtrsRay* rays, size_t n, PtrsHit* hits) {
  if (!scene || (n && (!rays || !hits))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  ON_DEVICE_OF(scene);
  DevBuf<PtrsRay> dr;
  DevBuf<PtrsHit> dh;
  CUDA_TRY(dr.upload(rays, n));
  CUDA_TRY(dh.alloc(n));
  int32_t rc = do_intersect(scene, dr.p, n, dh.p, nullptr, false, false, 0);
  if (rc != PTRS_OK) return rc;
  CUDA_TRY(cudaMemcpy(hits, dh.p, n * sizeof(PtrsHit), cudaMemcpyDeviceToHost));
  return PTRS_OK;
}
int32_t ptrs_intersect_p(PtrsScene* scene, const PtrsRay* rays, size_t n, uint8_t* occluded) {
  if (!scene || (n && (!rays || !occluded))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  ON_DEVICE_OF(scene);
  DevBuf<PtrsRay> dr;
  DevBuf<uint8_t> dh;
  CUDA_TRY(dr.upload(rays, n));
  CUDA_TRY(dh.alloc(n));
  int32_t rc = do_intersect(scene, dr.p, n, nullptr, dh.p, true, false, 0);
  if (rc != PTRS_OK) return rc;
  CUDA_TRY(cudaMemcpy(occluded, dh.p, n, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

// ---- film ----------------------------------------------------------------------------------------
int32_t ptrs_film_create(int32_t width, int32_t height, PtrsFilm** out) {
  if (!out || width <= 0 || height <= 0) return fail(PTRS_ERR_INVALID_ARGUMENT, "bad film size");
  std::unique_ptr<PtrsFilm> f(new PtrsFilm());
  f->width = width;
  f->height = height;
  f->owned = true;
  CUDA_TRY(cudaGetDevice(&f->device));
  // pooled, stream-ordered allocation like the scene buffers: creating / destroying a film per render does not
  // pay cudaMalloc / cudaFree (device-wide synchronisation, page mapping)
  CUDA_TRY(ptrs::pool_alloc(reinterpret_cast<void**>(&f->d), (size_t)width * height * sizeof(float4), (cudaStream_t)0));
  CUDA_TRY(cudaMemsetAsync(f->d, 0, (size_t)width * height * sizeof(float4), (cudaStream_t)0));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)0));
  *out = f.release();
  return PTRS_OK;
}
int32_t ptrs_film_wrap_device(int32_t width, int32_t height, float* d_rgbw, PtrsFilm** out) {
  if (!out || !d_rgbw || width <= 0 || height <= 0 || ((uintptr_t)d_rgbw & 15)) return fail(PTRS_ERR_INVALID_ARGUMENT, "bad film buffer (needs 16-byte alignment)");
  cudaPointerAttributes attr{};
  if (cudaPointerGetAttributes(&attr, d_rgbw) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(PTRS_ERR_INVALID_ARGUMENT, "film buffer is not device memory");
  }
  PtrsFilm* f = new PtrsFilm();
  f->device = attr.device;
  f->width = width;
  f->height = height;
  f->d = reinterpret_cast<float4*>(d_rgbw);
  f->owned = false;
  *out = f;
  return PTRS_OK;
}
int32_t ptrs_film_destroy(PtrsFilm* film) {
  if (!film) return PTRS_OK;
  ON_DEVICE_OF(film);
  if (film->owned && film->d) cudaFreeAsync(film->d, (cudaStream_t)0);
  delete film;
  return PTRS_OK;
}
int32_t ptrs_film_clear(PtrsFilm* film, void* stream) {
  if (!film) return fail(PTRS_ERR_INVALID_ARGUMENT, "null film");
  ON_DEVICE_OF(film);
  CUDA_TRY(cudaMemsetAsync(film->d, 0, (size_t)film->width * film->height * sizeof(float4), (cudaStream_t)stream));
  return PTRS_OK;
}
int32_t ptrs_film_download(PtrsFilm* film, float* rgbw) {
  if (!film || !rgbw) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  ON_DEVICE_OF(film);
  CUDA_TRY(cudaMemcpy(rgbw, film->d, (size_t)film->width * film->height * sizeof(float4), cudaMemcpyDeviceToHost));
  return PTRS_OK;
}
int32_t ptrs_film_resolve(PtrsFilm* film, float* rgb) {
  if (!film || !rgb) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  ON_DEVICE_OF(film);
  const uint32_t n = (uint32_t)film->width * film->height;
  DevBuf<float> d;
  CUDA_TRY(d.alloc((size_t)n * 3));
  launch_resolve(0, film->d, n, d.p, nullptr);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(rgb, d.p, (size_t)n * 12, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}
int32_t ptrs_film_resolve_srgb8(PtrsFilm* film, uint8_t* rgba) {
  if (!film || !rgba) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  ON_DEVICE_OF(film);
  const uint32_t n = (uint32_t)film->width * film->height;
  DevBuf<uint8_t> d;
  CUDA_TRY(d.alloc((size_t)n * 4));
  launch_resolve(0, film->d, n, nullptr, d.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(rgba, d.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}
float* ptrs_film_device_ptr(PtrsFilm* film) { return film ? reinterpret_cast<float*>(film->d) : nullptr; }

int32_t ptrs_film_sample_bounds(int32_t width, int32_t height, const float r[2], int32_t out[4]) {
  if (!r || !out) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  out[0] = (int)std::floor(0.5f - r[0]);
  out[1] = (int)std::floor(0.5f - r[1]);
  out[2] = (int)std::ceil((float)width - 0.5f + r[0]);
  out[3] = (int)std::ceil((float)height - 0.5f + r[1]);
  return PTRS_OK;
}

// One axis of ptrs_film_region_sample_rect.  A sample at position s has its film coordinate fx in [s, s + 1 - 2^-24]
// (the jitter is clamped to OneMinusEpsilon and the sum is rounded to float), and accumulate_kernel splats it onto
// pixels ceil(fx - 0.5 - r) .. floor(fx - 0.5 + r) + 1.  Both ends grow with fx, so position s reaches a pixel of
// [a, b) exactly when the footprint of its smallest fx starts below b and that of its largest fx ends above a.  The
// ends are evaluated with the kernel's float expressions, not with real-number bounds.
static void region_axis(int32_t sb0, int32_t sb1, float r, int32_t a, int32_t b, int32_t* lo, int32_t* hi) {
  *lo = sb1;
  *hi = sb0;
  for (int32_t s = sb0; s < sb1; ++s) {
    const float dx0 = (float)s - 0.5f, dx1 = ((float)s + 0x1.fffffep-1f) - 0.5f;
    const int p0 = (int)std::ceil(dx0 - r), p1 = (int)(std::floor(dx1 + r) + 1.0f);
    if (p0 < b && p1 > a) {
      *lo = std::min(*lo, s);
      *hi = std::max(*hi, s + 1);
    }
  }
}

int32_t ptrs_film_region_sample_rect(int32_t width, int32_t height, const float r[2], const int32_t pixel_rect[4], int32_t sample_rect[4]) {
  if (!r || !pixel_rect || !sample_rect) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (width <= 0 || height <= 0) return fail(PTRS_ERR_INVALID_ARGUMENT, "bad film resolution");
  if (!(r[0] > 0.f) || !(r[1] > 0.f) || !(r[0] < 1024.f) || !(r[1] < 1024.f)) return fail(PTRS_ERR_INVALID_ARGUMENT, "filter radius must be positive (and finite)");
  const int32_t size[2] = {width, height};
  for (int k = 0; k < 2; ++k)
    if (pixel_rect[k] < 0 || pixel_rect[k] >= pixel_rect[k + 2] || pixel_rect[k + 2] > size[k])
      return fail(PTRS_ERR_INVALID_ARGUMENT, "pixel rectangle empty, inverted or outside the film");
  int32_t sb[4];
  ptrs_film_sample_bounds(width, height, r, sb);
  int32_t out[4];
  for (int k = 0; k < 2; ++k) region_axis(sb[k], sb[k + 2], r[k], pixel_rect[k], pixel_rect[k + 2], &out[k], &out[k + 2]);
  std::memcpy(sample_rect, out, sizeof(out));
  return PTRS_OK;
}

// ---- integrator ----------------------------------------------------------------------------------
int32_t ptrs_render_params_default(PtrsRenderParams* p) {
  if (!p) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  std::memset(p, 0, sizeof(*p));
  p->spp = 1;
  p->max_depth = 15;
  p->rr_threshold = 1.0f;  // integrator.rs:240-242
  p->rr_start_depth = 3;
  p->rr_enable = 1;
  p->sample_stride = 1;
  p->filter_radius[0] = p->filter_radius[1] = 2.0f;  // GuassianFilter::new(2.), common/mod.rs:59, filter.rs:68-75
  const float alpha = 2.0f, radius = 2.0f;
  const float expv = std::exp(-alpha * radius * radius);
  int off = 0;
  for (int y = 0; y < 16; ++y)
    for (int x = 0; x < 16; ++x) {  // Film::new, film.rs:135-144
      float px = ((float)x + 0.5f) * radius / 16.0f, py = ((float)y + 0.5f) * radius / 16.0f;
      float gx = std::fmax(0.0f, std::exp(-alpha * px * px) - expv), gy = std::fmax(0.0f, std::exp(-alpha * py * py) - expv);
      p->filter_table[off++] = gx * gy;
    }
  return PTRS_OK;
}

static uint32_t default_paths_per_batch(PtrsScene* s) {
  if (const char* e = std::getenv("PTRS_PATHS_PER_BATCH")) {  // tuning override
    const long long v = std::atoll(e);
    if (v >= 32 && v <= (1ll << 30)) return (uint32_t)v;
  }
  if (s->default_cap == 0) {  // asked once per scene: cudaMemGetInfo is a slow call once the pools hold tens of GB
    uint64_t want = 1ull << 27;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      // the workspace this scene already holds counts as available
      const uint64_t avail = (uint64_t)free_b + s->ws.bytes();
      while (want > (1ull << 20) && want * Workspace::kBytesPerSlot > avail / 3) want >>= 1;
    }
    s->default_cap = (uint32_t)want;
  }
  return s->default_cap;
}

// sample_rect: the rectangle of sample positions to trace, {x0, y0, x1, y1} half-open, inside the sample bounds
// (ptrs_render passes the whole bounds); nullptr with a (pixel, sample number) list.
static int32_t render_impl(PtrsScene* s, const PtrsCamera* cam, const PtrsRenderParams* rp, PtrsFilm* film, const int32_t* sample_rect,
                           const int32_t* list_xy, const int32_t* list_s, size_t n_list, float* out_rgb, cudaStream_t st) {
  RenderConst rc;
  std::string why;
  int32_t r = build_render_const(cam, rp, &rc, &why);
  if (r != PTRS_OK) return fail(r, why);
  if (sample_rect) {
    for (int k = 0; k < 2; ++k) {
      const int32_t lo = sample_rect[k], hi = sample_rect[k + 2];
      if (lo >= hi || lo < rc.sb_min[k] || hi > rc.sb_min[k] + rc.sb_ext[k])
        return fail(PTRS_ERR_INVALID_ARGUMENT, "sample rectangle empty, inverted or outside the sample bounds");
      rc.rect_min[k] = lo;
      rc.rect_ext[k] = hi - lo;
    }
  }
  const uint32_t bw = ((uint32_t)rc.rect_ext[0] + 7u) >> 3, bh = ((uint32_t)rc.rect_ext[1] + 3u) >> 2;
  const uint64_t per_sample = (uint64_t)bw * bh * 32u;
  const uint64_t total = list_xy ? (uint64_t)n_list : per_sample * (uint64_t)rc.s_count;
  // Wavefront batch size.  Every batch pays for its tail: the rounds after Russian roulette has thinned the paths out are
  // latency-bound launches over nearly empty queues (on the 4K atrium ≈ 6.5 ms of an 89 ms batch of 16 Mi paths), so the
  // default is as large as the memory allows — 128 Mi slots x 368 B = 49 GB of the 180 GB — and never more than a third of
  // what is free on the device.
  uint32_t cap = rp->paths_per_batch > 0 ? (uint32_t)rp->paths_per_batch : ((uint64_t)s->ws.cap >= total && s->ws.cap > 0 ? s->ws.cap : default_paths_per_batch(s));
  cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>((cap + 31u) & ~31u, 32u), std::max<uint64_t>((total + 31) & ~31ull, 32));
  const uint32_t rounds = (uint32_t)rc.max_depth + 1 + 32;
  r = ensure_workspace(s, cap, rounds);
  if (r != PTRS_OK) return r;
  rc.cap = s->ws.cap;
  s->stats = PtrsStats{};
  r = ensure_split(s, &rc, st);
  if (r != PTRS_OK) return r;
  CUDA_TRY(cudaMemsetAsync(s->ws.gcount.p, 0, sizeof(GlobalCounters), st));
  DevBuf<int> d_xy, d_s;
  DevBuf<float4> d_dummy;
  if (list_xy) {
    r = check_pixel_list(rc, list_xy, list_s, n_list);
    if (r != PTRS_OK) return r;
    CUDA_TRY(d_xy.upload(list_xy, n_list * 2));
    CUDA_TRY(d_s.upload(list_s, n_list));
  }
  StageTimer tm{s, st};
  float ms[ST_COUNT] = {};
  uint64_t ext_rays = 0, paths = 0;
  CUDA_TRY(cudaEventRecord(s->ev[0], st));
  // equal batches (whole 8x4 blocks) rather than full ones and a remainder: a nearly empty last batch would
  // still pay for every round's launches
  const uint64_t n_batches = (total + s->ws.cap - 1) / s->ws.cap;
  const uint64_t per_batch = n_batches ? std::min<uint64_t>(s->ws.cap, (((total + n_batches - 1) / n_batches) + 31) & ~(uint64_t)31) : 0;
  for (uint64_t base = 0; base < total; base += per_batch) {
    const uint32_t n_work = (uint32_t)std::min<uint64_t>(per_batch, total - base);
    r = run_batch(s, rc, (rp->flags & PTRS_RENDER_EXACT_SHADING) != 0, base, n_work, list_xy ? d_xy.p + 2 * base : nullptr, list_xy ? d_s.p + base : nullptr, st, tm, &ext_rays);
    if (r != PTRS_OK) return r;
    if (film) {
      tm.begin(ST_ACCUMULATE);
      launch_accumulate(st, s->sm_count, rc, s->ws.arrays(), n_work, film->d);
      tm.end();
      s->stats.launches += 1;
    }
    if (out_rgb) {
      std::vector<float4> l(n_work);
      CUDA_TRY(cudaMemcpyAsync(l.data(), s->ws.L.p, (size_t)n_work * 16, cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      for (uint32_t i = 0; i < n_work; ++i) {
        out_rgb[3 * (base + i)] = l[i].x;
        out_rgb[3 * (base + i) + 1] = l[i].y;
        out_rgb[3 * (base + i) + 2] = l[i].z;
      }
    }
    s->stats.batches += 1;
  }
  CUDA_TRY(cudaEventRecord(s->ev[1], st));
  GlobalCounters g{};
  CUDA_TRY(cudaMemcpyAsync(&g, s->ws.gcount.p, sizeof(g), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  CUDA_TRY(cudaGetLastError());
  tm.collect(ms);
  float total_ms = 0.f;
  cudaEventElapsedTime(&total_ms, s->ev[0], s->ev[1]);
  // camera paths = valid (pixel, sample) pairs; 8x4 block padding outside the enumerated rectangle is not counted
  paths = list_xy ? n_list : (uint64_t)rc.rect_ext[0] * rc.rect_ext[1] * (uint64_t)rc.s_count;
  s->stats.camera_paths = paths;
  s->stats.extension_rays = ext_rays;
  s->stats.shadow_rays = g.shadow_rays;
  s->stats.mis_rays = g.mis_rays;
  s->stats.nodes_tested = g.nodes_tested;
  s->stats.tris_tested = g.tris_tested;
  s->stats.nee_nodes_tested = g.nee_nodes_tested;
  s->stats.nee_tris_tested = g.nee_tris_tested;
  s->stats.ms_generate = ms[ST_GENERATE];
  s->stats.ms_extend = ms[ST_EXTEND];
  s->stats.ms_shade = ms[ST_SHADE];
  s->stats.ms_shadow = ms[ST_CONNECT] + ms[ST_RESOLVE];
  s->stats.ms_connect_trace = ms[ST_CONNECT];
  s->stats.ms_resolve = ms[ST_RESOLVE];
  s->stats.ms_accumulate = ms[ST_ACCUMULATE];
  s->stats.ms_total = total_ms;
  return PTRS_OK;
}

int32_t ptrs_render_region(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t sample_rect[4], PtrsFilm* film,
                           void* stream) {
  if (!scene || !camera || !params || !sample_rect || !film) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (film->width != camera->width || film->height != camera->height) return fail(PTRS_ERR_INVALID_ARGUMENT, "film / camera resolution mismatch");
  if (film->device != scene->device) return fail(PTRS_ERR_INVALID_ARGUMENT, "film and scene live on different devices");
  ON_DEVICE_OF(scene);
  const int32_t r = render_impl(scene, camera, params, film, sample_rect, nullptr, nullptr, 0, nullptr, (cudaStream_t)stream);
  if (r != PTRS_OK) cudaStreamSynchronize((cudaStream_t)stream);  // nothing of the failed call may still run when its buffers are released
  return r;
}

int32_t ptrs_render(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params, PtrsFilm* film, void* stream) {
  if (!camera || !params) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  int32_t bounds[4];
  ptrs_film_sample_bounds(camera->width, camera->height, params->filter_radius, bounds);
  return ptrs_render_region(scene, camera, params, bounds, film, stream);
}

int32_t ptrs_path_radiance(PtrsScene* scene, const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t* pixels_xy,
                           const int32_t* sample_nums, size_t n, float* out_rgb) {
  if (!scene || !camera || !params || (n && (!pixels_xy || !sample_nums || !out_rgb))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  ON_DEVICE_OF(scene);
  const int32_t r = render_impl(scene, camera, params, nullptr, nullptr, pixels_xy, sample_nums, n, out_rgb, 0);
  if (r != PTRS_OK) cudaStreamSynchronize(0);
  return r;
}

int32_t ptrs_stats(const PtrsScene* scene, PtrsStats* out) {
  if (!scene || !out) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  *out = scene->stats;
  return PTRS_OK;
}
int32_t ptrs_set_stats_mode(PtrsScene* scene, int32_t count_visits) {
  if (!scene) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  scene->count_visits = count_visits != 0;
  return PTRS_OK;
}

// ---- parity probes ---------------------------------------------------------------------------------
int32_t ptrs_sobol_samples(const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t* pixels_xy, const int32_t* sample_nums,
                           size_t n, const int32_t* dims, size_t n_dims, float* out, uint64_t* out_index) {
  if (!camera || !params || (n && (!pixels_xy || !sample_nums || !dims || !out))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0 || n_dims == 0) return PTRS_OK;
  for (size_t k = 0; k < n_dims; ++k)
    if (dims[k] < 0 || dims[k] >= 1024) return fail(PTRS_ERR_INVALID_ARGUMENT, "dimension out of range");
  RenderConst rc;
  std::string why;
  int32_t r = build_render_const(camera, params, &rc, &why);
  if (r != PTRS_OK) return fail(r, why);
  const SobolHost& sh = sobol_host();
  DevBuf<uint32_t> tab;
  DevBuf<int> d_xy, d_s, d_dims;
  DevBuf<float> d_out;
  DevBuf<uint64_t> d_idx;
  CUDA_TRY(tab.upload(sh.matrices, (size_t)sh.n_dims * sh.n_cols));
  CUDA_TRY(d_xy.upload(pixels_xy, n * 2));
  CUDA_TRY(d_s.upload(sample_nums, n));
  CUDA_TRY(d_dims.upload(dims, n_dims));
  CUDA_TRY(d_out.alloc(n * n_dims));
  CUDA_TRY(d_idx.alloc(n));
  r = check_pixel_list(rc, pixels_xy, sample_nums, n);
  if (r != PTRS_OK) return r;
  if (plan_split(&rc) != PTRS_OK) return fail(PTRS_ERR_UNSUPPORTED, "resolution x max_depth too large for the Sobol split tables");
  DevBuf<uint32_t> split;
  r = build_split(&rc, tab.p, &split, 0);
  if (r != PTRS_OK) return r;
  // the draws as the render kernels make them (split tables) ...
  launch_sobol_probe(0, rc, tab.p, d_xy.p, d_s.p, (uint32_t)n, d_dims.p, (uint32_t)n_dims, d_out.p, d_idx.p, 0);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out, d_out.p, n * n_dims * 4, cudaMemcpyDeviceToHost));
  {  // ... which must be bit-identical to the reference's sobol_interval_to_index + sobol_sample on the device
    std::vector<float> generic(n * n_dims);
    launch_sobol_probe(0, rc, tab.p, d_xy.p, d_s.p, (uint32_t)n, d_dims.p, (uint32_t)n_dims, d_out.p, nullptr, 1);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(generic.data(), d_out.p, n * n_dims * 4, cudaMemcpyDeviceToHost));
    if (std::memcmp(generic.data(), out, n * n_dims * 4) != 0) return fail(PTRS_ERR_CUDA, "split-table Sobol draws differ from the generic path");
  }
  if (out_index) CUDA_TRY(cudaMemcpy(out_index, d_idx.p, n * 8, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

int32_t ptrs_generate_rays(const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t* pixels_xy, const int32_t* sample_nums,
                           size_t n, PtrsRay* rays, float* p_film, float* rxry_dir) {
  if (!camera || !params || (n && (!pixels_xy || !sample_nums || !rays))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  RenderConst rc;
  std::string why;
  int32_t r = build_render_const(camera, params, &rc, &why);
  if (r != PTRS_OK) return fail(r, why);
  const SobolHost& sh = sobol_host();
  DevBuf<uint32_t> tab;
  DevBuf<int> d_xy, d_s;
  DevBuf<PtrsRay> d_rays;
  DevBuf<float> d_pf, d_rx;
  CUDA_TRY(tab.upload(sh.matrices, (size_t)sh.n_dims * sh.n_cols));
  CUDA_TRY(d_xy.upload(pixels_xy, n * 2));
  CUDA_TRY(d_s.upload(sample_nums, n));
  CUDA_TRY(d_rays.alloc(n));
  CUDA_TRY(d_pf.alloc(n * 2));
  CUDA_TRY(d_rx.alloc(n * 6));
  r = check_pixel_list(rc, pixels_xy, sample_nums, n);
  if (r != PTRS_OK) return r;
  if (plan_split(&rc) != PTRS_OK) return fail(PTRS_ERR_UNSUPPORTED, "resolution x max_depth too large for the Sobol split tables");
  DevBuf<uint32_t> split;
  r = build_split(&rc, tab.p, &split, 0);
  if (r != PTRS_OK) return r;
  launch_ray_probe(0, rc, tab.p, d_xy.p, d_s.p, (uint32_t)n, d_rays.p, d_pf.p, d_rx.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(rays, d_rays.p, n * sizeof(PtrsRay), cudaMemcpyDeviceToHost));
  if (p_film) CUDA_TRY(cudaMemcpy(p_film, d_pf.p, n * 8, cudaMemcpyDeviceToHost));
  if (rxry_dir) CUDA_TRY(cudaMemcpy(rxry_dir, d_rx.p, n * 24, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

// ---- function-level probes (k_probe.cu) ------------------------------------------------------------------
static int32_t check_lobe(const PtrsLobeDesc* l) {
  if (l->kind < PTRS_LOBE_LAMBERTIAN || l->kind > PTRS_LOBE_DISNEY_DIFFUSE || l->fresnel < PTRS_FRESNEL_DIELECTRIC || l->fresnel > PTRS_FRESNEL_NOOP)
    return fail(PTRS_ERR_INVALID_ARGUMENT, "unknown lobe / Fresnel kind");
  return PTRS_OK;
}

int32_t ptrs_bxdf_eval(const PtrsLobeDesc* lobe, const float* wo, const float* wi, size_t n, int32_t flags, float* out) {
  if (!lobe || (n && (!wo || !wi || !out))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  if (n > 0x7fffffffull) return fail(PTRS_ERR_INVALID_ARGUMENT, "too many samples in one call");
  if (int32_t r = check_lobe(lobe)) return r;
  DevBuf<float> d_wo, d_wi, d_out;
  CUDA_TRY(d_wo.upload(wo, n * 3));
  CUDA_TRY(d_wi.upload(wi, n * 3));
  CUDA_TRY(d_out.alloc(n * 4));
  if (flags & PTRS_RENDER_EXACT_SHADING) launch_bxdf_eval_probe_exact(0, *lobe, d_wo.p, d_wi.p, (uint32_t)n, d_out.p);
  else launch_bxdf_eval_probe_fast(0, *lobe, d_wo.p, d_wi.p, (uint32_t)n, d_out.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out, d_out.p, n * 16, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

int32_t ptrs_bxdf_sample(const PtrsLobeDesc* lobe, const float* wo, const float* u, size_t n, int32_t flags, float* out) {
  if (!lobe || (n && (!wo || !u || !out))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return PTRS_OK;
  if (n > 0x7fffffffull) return fail(PTRS_ERR_INVALID_ARGUMENT, "too many samples in one call");
  if (int32_t r = check_lobe(lobe)) return r;
  DevBuf<float> d_wo, d_u, d_out;
  CUDA_TRY(d_wo.upload(wo, n * 3));
  CUDA_TRY(d_u.upload(u, n * 2));
  CUDA_TRY(d_out.alloc(n * 8));
  if (flags & PTRS_RENDER_EXACT_SHADING) launch_bxdf_sample_probe_exact(0, *lobe, d_wo.p, d_u.p, (uint32_t)n, d_out.p);
  else launch_bxdf_sample_probe_fast(0, *lobe, d_wo.p, d_u.p, (uint32_t)n, d_out.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out, d_out.p, n * 32, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

int32_t ptrs_light_sample(PtrsScene* scene, int32_t light, const float* ref_p, const float* ref_n, const float* u, size_t n, int32_t flags, float* out) {
  if (!scene || (n && (!ref_p || !ref_n || !u || !out))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (light < 0 || (uint32_t)light >= scene->dev.n_lights) return fail(PTRS_ERR_INVALID_ARGUMENT, "light index out of range");
  if (n == 0) return PTRS_OK;
  if (n > 0x7fffffffull) return fail(PTRS_ERR_INVALID_ARGUMENT, "too many samples in one call");
  ON_DEVICE_OF(scene);
  DevBuf<float> d_p, d_n, d_u, d_out;
  CUDA_TRY(d_p.upload(ref_p, n * 3));
  CUDA_TRY(d_n.upload(ref_n, n * 3));
  CUDA_TRY(d_u.upload(u, n * 2));
  CUDA_TRY(d_out.alloc(n * 16));
  if (flags & PTRS_RENDER_EXACT_SHADING) launch_light_sample_probe_exact(0, scene->dev, light, d_p.p, d_n.p, d_u.p, (uint32_t)n, d_out.p);
  else launch_light_sample_probe_fast(0, scene->dev, light, d_p.p, d_n.p, d_u.p, (uint32_t)n, d_out.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out, d_out.p, n * 64, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

int32_t ptrs_light_pdf(PtrsScene* scene, int32_t light, const float* ref_p, const float* ref_n, const float* wi, size_t n, int32_t flags, float* out) {
  if (!scene || (n && (!ref_p || !ref_n || !wi || !out))) return fail(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (light < 0 || (uint32_t)light >= scene->dev.n_lights) return fail(PTRS_ERR_INVALID_ARGUMENT, "light index out of range");
  if (n == 0) return PTRS_OK;
  if (n > 0x7fffffffull) return fail(PTRS_ERR_INVALID_ARGUMENT, "too many samples in one call");
  ON_DEVICE_OF(scene);
  DevBuf<float> d_p, d_n, d_w, d_out;
  CUDA_TRY(d_p.upload(ref_p, n * 3));
  CUDA_TRY(d_n.upload(ref_n, n * 3));
  CUDA_TRY(d_w.upload(wi, n * 3));
  CUDA_TRY(d_out.alloc(n));
  if (flags & PTRS_RENDER_EXACT_SHADING) launch_light_pdf_probe_exact(0, scene->dev, light, d_p.p, d_n.p, d_w.p, (uint32_t)n, d_out.p);
  else launch_light_pdf_probe_fast(0, scene->dev, light, d_p.p, d_n.p, d_w.p, (uint32_t)n, d_out.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out, d_out.p, n * 4, cudaMemcpyDeviceToHost));
  return PTRS_OK;
}

}  // extern "C"
