// Several GPUs of one node behind the C ABI (include/ptrs_b200.h, "Several GPUs of one node").
//
// The reference parallelises PathIntegrator::render over image tiles on the host's cores and merges every tile
// into the one film (integrator.rs:617-637, film.rs:213-228).  Across GPUs the unit of distribution is the Sobol
// sample number instead: the scene is replicated, device g of N renders the sample numbers s = g (mod N) of every
// pixel — the global Sobol index is a pure function of (pixel, sample number), sampler/sobol.rs:169-175, so the
// union over devices is exactly the reference's sample set and every device does the same amount of work — and the
// additive films (contrib_sum, filter_weight_sum are plain sums, film.rs:102-103) are combined by ONE collective,
// ncclReduce over NVLink, the only exchange step the path has.
//
// Two shapes:
//   PtrsMultiScene   one process drives all devices: one host thread, stream, scene replica and film per device,
//                    ncclCommInitAll; the reduce is issued for all devices from the calling thread in one NCCL group
//   PtrsComm         one process per GPU (torchrun / MPI style): ncclCommInitRank from an id the host ships around
// NCCL is bound at run time with dlopen, so the library has no link-time dependency on it and a process that
// already carries an NCCL (PyTorch) shares that copy instead of loading a second one.
#include <dlfcn.h>
#include <nccl.h>

#include <chrono>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "handles.hpp"

namespace {

using ptrs::set_error;

struct NcclApi {
  void* handle = nullptr;
  std::string why;
  decltype(&ncclGetVersion) GetVersion = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclReduce) Reduce = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok() const { return handle != nullptr; }
};

const NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[3] = {std::getenv("PTRS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    std::string tried;
    for (const char* n : names) {
      if (!n || !*n) continue;
      h = dlopen(n, RTLD_NOW | RTLD_LOCAL);
      if (h) break;
      tried += std::string(tried.empty() ? "" : "; ") + dlerror();
    }
    if (!h) {
      api.why = "NCCL is not loadable (" + tried + ")";
      return;
    }
    bool all = true;
    auto bind = [&](auto& fn, const char* sym) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, sym));
      if (!fn) {
        all = false;
        api.why = std::string("NCCL library lacks ") + sym;
      }
    };
    bind(api.GetVersion, "ncclGetVersion");
    bind(api.GetUniqueId, "ncclGetUniqueId");
    bind(api.CommInitRank, "ncclCommInitRank");
    bind(api.CommInitAll, "ncclCommInitAll");
    bind(api.CommDestroy, "ncclCommDestroy");
    bind(api.Reduce, "ncclReduce");
    bind(api.GroupStart, "ncclGroupStart");
    bind(api.GroupEnd, "ncclGroupEnd");
    bind(api.GetErrorString, "ncclGetErrorString");
    if (all) api.handle = h;
    else dlclose(h);
  });
  return api;
}

int32_t nccl_fail(const char* what, ncclResult_t r) {
  const NcclApi& a = nccl();
  return set_error(PTRS_ERR_NCCL, std::string(what) + ": " + (a.GetErrorString ? a.GetErrorString(r) : "NCCL error"));
}
#define NCCL_TRY(expr)                                   \
  do {                                                   \
    ncclResult_t r__ = (expr);                           \
    if (r__ != ncclSuccess) return nccl_fail(#expr, r__); \
  } while (0)
#define CUDA_TRY(expr)                                                                                              \
  do {                                                                                                              \
    cudaError_t e__ = (expr);                                                                                       \
    if (e__ != cudaSuccess) return set_error(PTRS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

// Communicators are per device LIST and live as long as the process: creating one costs hundreds of milliseconds and the
// first collective on it another second or so (NCCL connects lazily), which a host that re-creates its scene for every
// frame must not pay per frame.  `busy` serialises the collectives of handles that share an entry.
struct CommSet {
  std::vector<ncclComm_t> comm;
  std::mutex busy;
};
struct CommCache {
  std::mutex mu;
  std::map<std::vector<int>, std::unique_ptr<CommSet>> sets;
};
CommCache& comm_cache() {
  static CommCache* c = new CommCache();  // intentionally not destroyed: NCCL may already be unloading at exit
  return *c;
}

struct DeviceScope {  // the calling thread's current device is restored on exit
  int prev = -1;
  explicit DeviceScope(int dev) {
    cudaGetDevice(&prev);
    cudaSetDevice(dev);
  }
  ~DeviceScope() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace

struct PtrsComm {
  int device = 0;
  ncclComm_t comm = nullptr;
  int n_ranks = 1, rank = 0;
};

struct PtrsMultiScene {
  int n = 0;
  std::vector<int> device;
  std::vector<PtrsScene*> scene;
  std::vector<PtrsFilm*> film;
  std::vector<cudaStream_t> stream;
  CommSet* comms = nullptr;  // null when n == 1; owned by the process-wide cache
  int film_w = 0, film_h = 0;
  ~PtrsMultiScene() {
    for (int g = 0; g < n; ++g) {
      DeviceScope on(device[g]);
      if (g < (int)stream.size() && stream[g]) cudaStreamSynchronize(stream[g]);
      if (g < (int)film.size() && film[g]) ptrs_film_destroy(film[g]);
      if (g < (int)scene.size() && scene[g]) ptrs_scene_destroy(scene[g]);
      if (g < (int)stream.size() && stream[g]) cudaStreamDestroy(stream[g]);
    }
  }
};

namespace {

// run fn(g) for every device index on its own host thread (the calling thread takes g = 0); the first failure
// (lowest g) becomes the calling thread's error
template <class F>
int32_t for_each_device(const PtrsMultiScene& m, F fn) {
  std::vector<int32_t> rc(m.n, PTRS_OK);
  std::vector<std::string> msg(m.n);
  auto body = [&](int g) {
    DeviceScope on(m.device[g]);
    rc[g] = fn(g);
    if (rc[g] != PTRS_OK) msg[g] = ptrs_last_error();
  };
  std::vector<std::thread> th;
  for (int g = 1; g < m.n; ++g) th.emplace_back(body, g);
  body(0);
  for (auto& t : th) t.join();
  for (int g = 0; g < m.n; ++g)
    if (rc[g] != PTRS_OK) return set_error(rc[g], "device " + std::to_string(m.device[g]) + ": " + msg[g]);
  return PTRS_OK;
}

int32_t ensure_films(PtrsMultiScene* m, int w, int h) {
  if (m->film_w == w && m->film_h == h && (int)m->film.size() == m->n) return PTRS_OK;
  for (int g = 0; g < (int)m->film.size(); ++g)
    if (m->film[g]) {
      DeviceScope on(m->device[g]);
      ptrs_film_destroy(m->film[g]);
    }
  m->film.assign(m->n, nullptr);
  m->film_w = m->film_h = 0;
  const int32_t r = for_each_device(*m, [&](int g) { return ptrs_film_create(w, h, &m->film[g]); });
  if (r != PTRS_OK) return r;
  m->film_w = w;
  m->film_h = h;
  return PTRS_OK;
}

}  // namespace

extern "C" {

int32_t ptrs_multi_create(const PtrsSceneDesc* desc, int32_t n_devices, const int32_t* devices, int32_t device_bvh, PtrsMultiScene** out) {
  if (!desc || !out || n_devices < 1 || n_devices > 64) return set_error(PTRS_ERR_INVALID_ARGUMENT, "bad argument");
  int avail = 0;
  CUDA_TRY(cudaGetDeviceCount(&avail));
  std::unique_ptr<PtrsMultiScene> m(new PtrsMultiScene());
  for (int g = 0; g < n_devices; ++g) {
    const int d = devices ? devices[g] : g;
    if (d < 0 || d >= avail) return set_error(PTRS_ERR_INVALID_ARGUMENT, "device index out of range (" + std::to_string(avail) + " visible)");
    for (int k : m->device)
      if (k == d) return set_error(PTRS_ERR_INVALID_ARGUMENT, "a device is listed twice");
    m->device.push_back(d);
  }
  m->n = n_devices;
  if (n_devices > 1 && !nccl().ok()) return set_error(PTRS_ERR_NCCL, nccl().why);
  m->scene.assign(n_devices, nullptr);
  m->stream.assign(n_devices, nullptr);
  int32_t r = for_each_device(*m, [&](int g) -> int32_t {
    const int32_t rc = device_bvh ? ptrs_scene_create_device_bvh(desc, &m->scene[g]) : ptrs_scene_create(desc, &m->scene[g]);
    if (rc != PTRS_OK) return rc;
    CUDA_TRY(cudaStreamCreate(&m->stream[g]));
    return PTRS_OK;
  });
  if (r != PTRS_OK) return r;
  if (n_devices > 1) {
    CommCache& cache = comm_cache();
    std::lock_guard<std::mutex> lock(cache.mu);
    std::unique_ptr<CommSet>& slot = cache.sets[m->device];
    if (!slot) {
      std::unique_ptr<CommSet> cs(new CommSet());
      cs->comm.assign(n_devices, nullptr);
      NCCL_TRY(nccl().CommInitAll(cs->comm.data(), n_devices, m->device.data()));
      slot = std::move(cs);
    }
    m->comms = slot.get();
  }
  *out = m.release();
  return PTRS_OK;
}

int32_t ptrs_multi_destroy(PtrsMultiScene* multi) {
  delete multi;
  return PTRS_OK;
}

int32_t ptrs_multi_device_count(const PtrsMultiScene* multi, int32_t* n_devices) {
  if (!multi || !n_devices) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  *n_devices = multi->n;
  return PTRS_OK;
}

int32_t ptrs_multi_root_film(PtrsMultiScene* multi, PtrsFilm** film) {
  if (!multi || !film) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (multi->film.empty() || !multi->film[0]) return set_error(PTRS_ERR_INVALID_ARGUMENT, "nothing rendered yet");
  *film = multi->film[0];
  return PTRS_OK;
}

int32_t ptrs_multi_scene(PtrsMultiScene* multi, int32_t g, PtrsScene** scene) {
  if (!multi || !scene || g < 0 || g >= multi->n) return set_error(PTRS_ERR_INVALID_ARGUMENT, "bad argument");
  *scene = multi->scene[g];
  return PTRS_OK;
}

int32_t ptrs_multi_render_region(PtrsMultiScene* multi, const PtrsCamera* camera, const PtrsRenderParams* params, const int32_t sample_rect[4],
                                 float* host_rgbw, PtrsStats* per_device_stats, float* total_ms) {
  if (!multi || !camera || !params || !sample_rect) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  const auto t0 = std::chrono::steady_clock::now();
  PtrsMultiScene& m = *multi;
  int32_t r = ensure_films(&m, camera->width, camera->height);
  if (r != PTRS_OK) return r;
  // shard g of the caller's own selection: the caller's (stride, phase) picks s = phase (mod stride); of those,
  // device g takes every n-th
  const int stride = params->sample_stride > 0 ? params->sample_stride : 1;
  const int phase = ((params->sample_phase % stride) + stride) % stride;
  r = for_each_device(m, [&](int g) -> int32_t {
    int32_t rc = ptrs_film_clear(m.film[g], m.stream[g]);
    if (rc != PTRS_OK) return rc;
    PtrsRenderParams p = *params;
    p.sample_stride = stride * m.n;
    p.sample_phase = phase + g * stride;
    rc = ptrs_render_region(m.scene[g], camera, &p, sample_rect, m.film[g], m.stream[g]);
    if (rc != PTRS_OK) return rc;
    if (per_device_stats) rc = ptrs_stats(m.scene[g], per_device_stats + g);
    return rc;
  });
  if (r != PTRS_OK) return r;
  if (m.n > 1) {
    // every device's render has been enqueued and joined: the reduce of all devices goes out as one NCCL group from
    // this thread (the single-thread multi-device pattern), each part ordered on its device's stream
    const size_t count = (size_t)m.film_w * m.film_h * 4;
    std::lock_guard<std::mutex> one_collective_at_a_time(m.comms->busy);
    NCCL_TRY(nccl().GroupStart());
    for (int g = 0; g < m.n; ++g) {
      const ncclResult_t nr = nccl().Reduce(m.film[g]->d, m.film[g]->d, count, ncclFloat32, ncclSum, 0, m.comms->comm[g], m.stream[g]);
      if (nr != ncclSuccess) {
        nccl().GroupEnd();
        return nccl_fail("ncclReduce", nr);
      }
    }
    NCCL_TRY(nccl().GroupEnd());
    for (int g = 0; g < m.n; ++g) {
      DeviceScope on(m.device[g]);
      CUDA_TRY(cudaStreamSynchronize(m.stream[g]));
    }
  }
  if (host_rgbw) {
    DeviceScope on(m.device[0]);
    CUDA_TRY(cudaMemcpyAsync(host_rgbw, m.film[0]->d, (size_t)m.film_w * m.film_h * 16, cudaMemcpyDeviceToHost, m.stream[0]));
    CUDA_TRY(cudaStreamSynchronize(m.stream[0]));
  }
  if (total_ms) *total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return PTRS_OK;
}

int32_t ptrs_multi_render(PtrsMultiScene* multi, const PtrsCamera* camera, const PtrsRenderParams* params, float* host_rgbw, PtrsStats* per_device_stats,
                          float* total_ms) {
  if (!camera || !params) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  int32_t bounds[4];
  ptrs_film_sample_bounds(camera->width, camera->height, params->filter_radius, bounds);
  return ptrs_multi_render_region(multi, camera, params, bounds, host_rgbw, per_device_stats, total_ms);
}

// ---- one process per GPU ---------------------------------------------------------------------------------
int32_t ptrs_comm_unique_id(uint8_t id[PTRS_COMM_ID_BYTES]) {
  static_assert(PTRS_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
  if (!id) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (!nccl().ok()) return set_error(PTRS_ERR_NCCL, nccl().why);
  ncclUniqueId u;
  NCCL_TRY(nccl().GetUniqueId(&u));
  std::memcpy(id, u.internal, NCCL_UNIQUE_ID_BYTES);
  return PTRS_OK;
}

int32_t ptrs_comm_init_rank(const uint8_t id[PTRS_COMM_ID_BYTES], int32_t n_ranks, int32_t rank, PtrsComm** out) {
  if (!id || !out || n_ranks < 1 || rank < 0 || rank >= n_ranks) return set_error(PTRS_ERR_INVALID_ARGUMENT, "bad argument");
  if (!nccl().ok()) return set_error(PTRS_ERR_NCCL, nccl().why);
  std::unique_ptr<PtrsComm> c(new PtrsComm());
  CUDA_TRY(cudaGetDevice(&c->device));
  ncclUniqueId u;
  std::memcpy(u.internal, id, NCCL_UNIQUE_ID_BYTES);
  NCCL_TRY(nccl().CommInitRank(&c->comm, n_ranks, u, rank));
  c->n_ranks = n_ranks;
  c->rank = rank;
  *out = c.release();
  return PTRS_OK;
}

int32_t ptrs_comm_destroy(PtrsComm* comm) {
  if (!comm) return PTRS_OK;
  if (comm->comm) {
    DeviceScope on(comm->device);
    nccl().CommDestroy(comm->comm);
  }
  delete comm;
  return PTRS_OK;
}

int32_t ptrs_comm_info(const PtrsComm* comm, int32_t* n_ranks, int32_t* rank) {
  if (!comm) return set_error(PTRS_ERR_INVALID_ARGUMENT, "null argument");
  if (n_ranks) *n_ranks = comm->n_ranks;
  if (rank) *rank = comm->rank;
  return PTRS_OK;
}

int32_t ptrs_film_reduce(PtrsComm* comm, PtrsFilm* film, int32_t root, void* stream) {
  if (!comm || !film || root < 0 || root >= comm->n_ranks) return set_error(PTRS_ERR_INVALID_ARGUMENT, "bad argument");
  if (film->device != comm->device) return set_error(PTRS_ERR_INVALID_ARGUMENT, "film and communicator live on different devices");
  DeviceScope on(comm->device);
  NCCL_TRY(nccl().Reduce(film->d, film->d, (size_t)film->width * film->height * 4, ncclFloat32, ncclSum, root, comm->comm, (cudaStream_t)stream));
  return PTRS_OK;
}

}  // extern "C"
