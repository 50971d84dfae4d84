// C++ mirror of the reference's host-facing interface for the rendering path, over the C ABI
// (include/ptrs_b200.h).  Same names, argument meaning and call order as the Rust API it stands in for:
//
//   SamplerBuilder::new(log, spp, &sample_bounds)            src/pathtracer/sampler/sobol.rs:35
//   PathIntegrator::new(log, sampler_builder, max_depth, ..) src/pathtracer/integrator.rs:230
//   PathIntegrator::preprocess(&RenderScene)                 src/pathtracer/integrator.rs:250
//   PathIntegrator::render(&self, &Camera, &RenderScene)     src/pathtracer/integrator.rs:536
//   RenderScene::{intersect, intersect_p, world_bound}       src/pathtracer/mod.rs:92-102
//   Film::{clear, get_sample_bounds, to_rgba_image, to_channel_updates}   src/common/film.rs:164-271
//   Camera { .., film }                                      src/common/mod.rs:19-62
//
// Error behaviour: the reference panics on unsupported input and logs numeric anomalies; here every
// failing C-ABI call throws ptrs::Error carrying the status code and ptrs_last_error().
#pragma once
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ptrs_b200.h"
#include "scene_builder.hpp"

namespace ptrs {

struct Error : std::runtime_error {
  int32_t code;
  Error(int32_t c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int32_t rc) {
  if (rc != PTRS_OK) throw Error(rc, ptrs_last_error());
}

struct Bounds2i {
  int32_t x0, y0, x1, y1;
};

class Film {
 public:
  Film(int32_t width, int32_t height) : w_(width), h_(height) { check(ptrs_film_create(width, height, &f_)); }
  ~Film() { ptrs_film_destroy(f_); }
  Film(const Film&) = delete;
  Film& operator=(const Film&) = delete;
  void clear() { check(ptrs_film_clear(f_, nullptr)); }                                  // film.rs:164-172
  Bounds2i get_sample_bounds(const float radius[2]) const {                              // film.rs:174-185
    int32_t b[4];
    check(ptrs_film_sample_bounds(w_, h_, radius, b));
    return Bounds2i{b[0], b[1], b[2], b[3]};
  }
  // the sample rectangle whose render completes the pixels of pixel_rect (ptrs_film_region_sample_rect)
  Bounds2i region_sample_rect(const Bounds2i& pixel_rect, const float radius[2]) const {
    const int32_t p[4] = {pixel_rect.x0, pixel_rect.y0, pixel_rect.x1, pixel_rect.y1};
    int32_t b[4];
    check(ptrs_film_region_sample_rect(w_, h_, radius, p, b));
    return Bounds2i{b[0], b[1], b[2], b[3]};
  }
  std::vector<uint8_t> to_rgba_image() const {                                           // film.rs:230-251
    std::vector<uint8_t> out((size_t)w_ * h_ * 4);
    check(ptrs_film_resolve_srgb8(f_, out.data()));
    return out;
  }
  std::array<std::vector<float>, 3> to_channel_updates() const {                         // film.rs:253-271
    std::vector<float> rgb((size_t)w_ * h_ * 3);
    check(ptrs_film_resolve(f_, rgb.data()));
    std::array<std::vector<float>, 3> ch;
    for (auto& c : ch) c.resize((size_t)w_ * h_);
    for (size_t i = 0; i < (size_t)w_ * h_; ++i)
      for (int k = 0; k < 3; ++k) ch[k][i] = rgb[3 * i + k];
    return ch;
  }
  int32_t width() const { return w_; }
  int32_t height() const { return h_; }
  PtrsFilm* handle() const { return f_; }

 private:
  int32_t w_, h_;
  PtrsFilm* f_ = nullptr;
};

// Camera owns its Film like the reference's (common/mod.rs:19-30).
struct Camera {
  PtrsCamera cam;
  Film film;
  explicit Camera(const PtrsCamera& c) : cam(c), film(c.width, c.height) {}
};

class RenderScene {
 public:
  explicit RenderScene(const ptrs_host::FlatScene& flat) : n_lights_(flat.lights.size()) {
    PtrsSceneDesc d = flat.desc();
    check(ptrs_scene_create(&d, &s_));
  }
  ~RenderScene() { ptrs_scene_destroy(s_); }
  RenderScene(const RenderScene&) = delete;
  RenderScene& operator=(const RenderScene&) = delete;
  // mod.rs:92-94: on a hit, r.t_max is shortened like GeometricPrimitive::intersect does (primitive.rs:48)
  bool intersect(PtrsRay& r, PtrsHit& isect) const {
    check(ptrs_intersect(s_, &r, 1, &isect));
    if (isect.prim < 0) return false;
    r.t_max = isect.t;
    return true;
  }
  bool intersect_p(const PtrsRay& r) const {  // mod.rs:96-98
    uint8_t occ = 0;
    check(ptrs_intersect_p(s_, &r, 1, &occ));
    return occ != 0;
  }
  void intersect(const std::vector<PtrsRay>& rays, std::vector<PtrsHit>& hits) const {
    hits.resize(rays.size());
    check(ptrs_intersect(s_, rays.data(), rays.size(), hits.data()));
  }
  ptrs_host::Bounds3 world_bound() const {  // mod.rs:100-102
    float b[6];
    check(ptrs_scene_world_bound(s_, b));
    return ptrs_host::Bounds3{{b[0], b[1], b[2]}, {b[3], b[4], b[5]}};
  }
  size_t n_lights() const { return n_lights_; }
  PtrsScene* handle() const { return s_; }

 private:
  PtrsScene* s_ = nullptr;
  size_t n_lights_;
};

class SamplerBuilder {  // SobolSamplerBuilder
 public:
  SamplerBuilder(size_t samples_per_pixel, const Bounds2i& sample_bounds) : spp_(samples_per_pixel), bounds_(sample_bounds) {}
  SamplerBuilder& with_seed(uint64_t) { return *this; }  // ignored, like sobol.rs:75-77
  size_t samples_per_pixel() const { return spp_; }

 private:
  size_t spp_;
  Bounds2i bounds_;
};

class PathIntegrator {
 public:
  PathIntegrator(const SamplerBuilder& sb, int32_t max_depth, bool show_progress_bar = false) : progress_(show_progress_bar) {
    check(ptrs_render_params_default(&params_));  // rr_threshold 1.0, rr_start_depth 3, rr_enable (integrator.rs:240-242)
    params_.spp = (int32_t)sb.samples_per_pixel();
    params_.max_depth = max_depth;
  }
  void preprocess(const RenderScene& scene) { too_many_lights_ = scene.n_lights() > 16; }  // integrator.rs:250-258
  void toggle_progress_bar() { progress_ = !progress_; }
  void render(Camera& camera, const RenderScene& scene) const {  // integrator.rs:536: accumulates into camera.film
    check(ptrs_render(scene.handle(), &camera.cam, &params_, camera.film.handle(), nullptr));
  }
  // the same restricted to a rectangle of sample positions (ptrs_render_region), e.g. one tile of integrator.rs:545-637
  void render(Camera& camera, const RenderScene& scene, const Bounds2i& sample_rect) const {
    const int32_t r[4] = {sample_rect.x0, sample_rect.y0, sample_rect.x1, sample_rect.y1};
    check(ptrs_render_region(scene.handle(), &camera.cam, &params_, r, camera.film.handle(), nullptr));
  }
  PtrsStats stats(const RenderScene& scene) const {
    PtrsStats st;
    check(ptrs_stats(scene.handle(), &st));
    return st;
  }
  PtrsRenderParams& params() { return params_; }
  bool too_many_lights() const { return too_many_lights_; }

 private:
  PtrsRenderParams params_;
  bool progress_, too_many_lights_ = false;
};

}  // namespace ptrs
