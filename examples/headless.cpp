// Stand-in for the reference's headless CLI on top of the C ABI (src/main.rs:37-148, src/headless.rs:180-234):
//   headless SCENE -o OUTDIR [-s SAMPLES] [-r WxH] [-d MAX_DEPTH] [--server HOST:PORT] [--default_lights]
//            [--sunsky-hdr FILE] [--crop X0,Y0,X1,Y1]
// imports SCENE (.xml / .gltf / .glb), renders it on the GPU and writes OUTDIR/render.png.  --crop renders only the
// pixel rectangle [X0, X1) x [Y0, Y1) of the image, exactly as the full render has it, and writes (and streams) an
// image of the crop's size.  When a tev display
// server answers at --server the film is streamed to it every 2 s while the render runs in sample passes
// (the reference reads its film concurrently under an RwLock; here the preview thread reads between passes).
#include <array>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../pathtracer_rs_b200/host/image_io.hpp"
#include "../pathtracer_rs_b200/host/importers.hpp"
#include "../pathtracer_rs_b200/host/pathtracer.hpp"
#include "../pathtracer_rs_b200/host/tev.hpp"

static bool parse_resolution(const char* s, int* w, int* h) {  // main.rs:22-34
  float x, y;
  if (std::sscanf(s, "%fx%f", &x, &y) != 2) return false;
  *w = (int)x;
  *h = (int)y;
  return *w > 0 && *h > 0;
}

static bool parse_crop(const char* s, ptrs::Bounds2i* c) {
  return std::sscanf(s, "%d,%d,%d,%d", &c->x0, &c->y0, &c->x1, &c->y1) == 4;
}

// rows [y0, y1) x columns [x0, x1) of a row-major image of `width` pixels with `n` values each
template <typename T>
static std::vector<T> crop_image(const std::vector<T>& img, int width, int n, const ptrs::Bounds2i& c) {
  std::vector<T> out;
  out.reserve((size_t)(c.x1 - c.x0) * (c.y1 - c.y0) * n);
  for (int y = c.y0; y < c.y1; ++y)
    out.insert(out.end(), img.begin() + ((size_t)y * width + c.x0) * n, img.begin() + ((size_t)y * width + c.x1) * n);
  return out;
}

static void stream_film(ptrs_host::TevClient& tev, const ptrs::Film& film, const ptrs::Bounds2i& crop) {
  const auto ch = film.to_channel_updates();
  std::array<std::vector<float>, 3> cropped;
  for (int k = 0; k < 3; ++k) cropped[k] = crop_image(ch[k], film.width(), 1, crop);
  const float* planes[3] = {cropped[0].data(), cropped[1].data(), cropped[2].data()};
  for (const auto& m : ptrs_host::tev_update_image(planes, crop.x1 - crop.x0, crop.y1 - crop.y0, "render"))
    if (!tev.send(m)) return;
}

int main(int argc, char** argv) {
  std::string scene_path, out_dir, server = "127.0.0.1:14158";
  ptrs_host::ImportOptions opt;
  int spp = 1, max_depth = 15;
  bool has_crop = false;
  ptrs::Bounds2i crop{};
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    auto val = [&]() -> const char* { return i + 1 < argc ? argv[++i] : ""; };
    if (a == "-o" || a == "--output") out_dir = val();
    else if (a == "-s" || a == "--samples") spp = std::atoi(val());
    else if (a == "-r" || a == "--resolution") {
      if (!parse_resolution(val(), &opt.res_w, &opt.res_h)) std::fprintf(stderr, "failed parsing resolution string, falling back to default resolution\n");
    } else if (a == "-d" || a == "--max_depth") max_depth = std::atoi(val());
    else if (a == "--server") server = val();
    else if (a == "--default_lights") opt.default_lights = true;
    else if (a == "--sunsky-hdr") opt.sunsky_hdr = val();
    else if (a == "--crop") {
      if (!parse_crop(val(), &crop)) {
        std::fprintf(stderr, "--crop wants X0,Y0,X1,Y1\n");
        return 2;
      }
      has_crop = true;
    } else if (a == "--headless") {}
    else if (a[0] != '-') scene_path = a;
  }
  if (scene_path.empty() || out_dir.empty()) {
    std::fprintf(stderr, "usage: headless SCENE -o OUTDIR [-s SAMPLES] [-r WxH] [-d MAX_DEPTH] [--server HOST:PORT] [--crop X0,Y0,X1,Y1]\n");
    return 2;
  }
  try {
    ptrs_host::SceneBuilder builder;
    const PtrsCamera cam = ptrs_host::import_scene(scene_path, opt, builder);
    const ptrs_host::FlatScene flat = builder.finalize(4);
    ptrs::Camera camera(cam);
    ptrs::RenderScene scene(flat);
    const float radius[2] = {2.f, 2.f};
    ptrs::SamplerBuilder sampler((size_t)spp, camera.film.get_sample_bounds(radius));
    ptrs::PathIntegrator integrator(sampler, max_depth, true);
    integrator.preprocess(scene);
    if (!has_crop) crop = ptrs::Bounds2i{0, 0, cam.width, cam.height};
    // the sample positions whose filter footprints reach the crop: rendering them completes its pixels
    const ptrs::Bounds2i sample_rect = camera.film.region_sample_rect(crop, radius);
    const int crop_w = crop.x1 - crop.x0, crop_h = crop.y1 - crop.y0;
    ptrs_host::TevClient tev;
    const auto t0 = std::chrono::steady_clock::now();
    if (tev.connect(server)) {
      tev.send(ptrs_host::tev_create_image(crop_w, crop_h, "render"));
      // sample passes of at most 16 spp each; the film is additive, so the union of the passes is the full render
      int spp2 = 1;
      while (spp2 < spp) spp2 <<= 1;
      auto last = std::chrono::steady_clock::now();
      for (int s0 = 0; s0 < spp2; s0 += 16) {
        integrator.params().sample_begin = s0;
        integrator.params().sample_end = std::min(spp2, s0 + 16);
        integrator.render(camera, scene, sample_rect);
        if (std::chrono::steady_clock::now() - last >= std::chrono::seconds(2)) {
          stream_film(tev, camera.film, crop);
          last = std::chrono::steady_clock::now();
        }
      }
      stream_film(tev, camera.film, crop);
    } else {
      std::fprintf(stderr, "could not connect to display server, falling back to one shot rendering\n");
      integrator.render(camera, scene, sample_rect);
    }
    const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    const PtrsStats st = integrator.stats(scene);
    std::printf("rendering took: %.3f s (%u triangles, %u x %u, %d spp, last pass %.1f M samples/s)\n", sec, (unsigned)flat.prim_vertex.size() / 3,
                (unsigned)crop_w, (unsigned)crop_h, spp, st.camera_paths / st.ms_total / 1e3);
    const std::vector<uint8_t> img = crop_image(camera.film.to_rgba_image(), cam.width, 4, crop);
    const std::string out = out_dir + "/render.png";  // main.rs:66
    ptrs_host::save_png(out, img.data(), crop_w, crop_h, 4);
    std::printf("wrote %s\n", out.c_str());
  } catch (const ptrs::Error& e) {
    std::fprintf(stderr, "ptrs error %d: %s\n", e.code, e.what());
    return 1;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 1;
  }
  return 0;
}
