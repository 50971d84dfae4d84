// generate / shade_miss / accumulate / resolve / parity-probe kernels
#include <algorithm>

#include "launch.hpp"
#include "wavefront.cuh"

namespace ptrs {

// ---- generate --------------------------------------------------------------------------------------
// Work item w of a batch -> (sample j, pixel).  Pixels of the enumerated rectangle are visited in 8x4 blocks
// so that a warp covers a compact screen tile (coherent primary rays); samples are the slow index.
PT_DEV void work_to_pixel(const RenderConst& rc, uint64_t w, int* px, int* py, int* sample) {
  const uint32_t bw = ((uint32_t)rc.rect_ext[0] + 7u) >> 3, bh = ((uint32_t)rc.rect_ext[1] + 3u) >> 2;
  const uint64_t per_sample = (uint64_t)bw * bh * 32u;
  const uint32_t j = (uint32_t)(w / per_sample);
  const uint32_t r = (uint32_t)(w % per_sample);
  const uint32_t blk = r >> 5, in = r & 31u;
  const uint32_t bx = blk % bw, by = blk / bw;
  *px = rc.rect_min[0] + (int)(bx * 8u + (in & 7u));
  *py = rc.rect_min[1] + (int)(by * 4u + (in >> 3));
  *sample = rc.s_begin + (int)j * rc.s_stride;
}

__global__ void __launch_bounds__(256) generate_kernel(const __grid_constant__ RenderConst rc, const uint32_t* __restrict__ sobol,
                                                        PathArrays P, uint64_t work_base, uint32_t n_work, const int* __restrict__ list_xy,
                                                        const int* __restrict__ list_s, int* __restrict__ q_ext, RoundCounters* ctr) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ((n_work + 31u) & ~31u); i += stride) {
    bool valid = i < n_work;
    int px = 0, py = 0, s = 0;
    if (valid) {
      if (list_xy) {
        px = list_xy[2 * i];
        py = list_xy[2 * i + 1];
        s = list_s[i];
      } else {
        work_to_pixel(rc, work_base + i, &px, &py, &s);
        valid = px < rc.rect_min[0] + rc.rect_ext[0] && py < rc.rect_min[1] + rc.rect_ext[1];
      }
    }
    if (valid) {
      PathSampler ps;
      sampler_start(rc.sobol, rc.split, ps, px, py, (uint32_t)s, 0u);
      V2 u = get_2d(rc.sobol, rc.split, sobol, ps);
      const float fx = (float)px + u.x, fy = (float)py + u.y;  // get_camera_sample, sobol.rs:116-120
      V3 o, d;
      camera_ray(rc.cam, fx, fy, rc.diff_scale, &o, &d, nullptr, nullptr);
      PathRay r;
      r.ox = o.x;
      r.oy = o.y;
      r.oz = o.z;
      r.packed = pack_state(ps.dimension | PT_F_HAS_DIFF, 0);
      r.dx = d.x;
      r.dy = d.y;
      r.dz = d.z;
      r.eta_scale = 1.f;
      PathAux a;
      a.br = a.bg = a.bb = 1.f;
      a.pixel = pack_pixel(px, py);
      a.sample = (uint32_t)s;
      a.spare = 0u;
      a.fx = fx;
      a.fy = fy;
      st256(&P.slot[i].r, r);
      st256(&P.slot[i].a, a);
      P.L[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else if (i < n_work) {
      PathAux a;
      a.br = a.bg = a.bb = 0.f;
      a.pixel = 0u;
      a.sample = 0u;
      a.spare = 0u;
      a.fx = a.fy = -1e30f;  // padding lane of an 8x4 block outside the enumerated rectangle
      st256(&P.slot[i].a, a);
      P.L[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    warp_push(valid, i, q_ext, &ctr->n_ext);
  }
}

// ---- shade -----------------------------------------------------------------------------------------
// "miss" class: Σ infinite lights Le for camera / specular paths, then the path ends (integrator.rs:418-431)
__global__ void __launch_bounds__(128) shade_miss_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ PathArrays P, const int* __restrict__ q, RoundCounters* ctr) {
  const uint32_t n = ctr->n_class[PT_CLASS_MISS];
  const int lane = threadIdx.x & 31;
  for (;;) {
    const uint32_t base = warp_fetch32(&ctr->t_class[PT_CLASS_MISS]);
    if (base >= n) break;
    const uint32_t i = base + lane;
    if (i >= n) continue;
    const int p = q[i];
    const PathRay r = ld256(&P.slot[p].r);
    if (packed_bounces(r.packed) == 0 || (r.packed & PT_F_SPECULAR)) {
      const PathAux a = ld256(&P.slot[p].a);
      float4 l4 = P.L[p];
      const V3 d = mk3(r.dx, r.dy, r.dz);
      Spec l = sp(l4.x, l4.y, l4.z), beta = sp(a.br, a.bg, a.bb);
      for (uint32_t k = 0; k < sc.n_infinite_lights; ++k) l = l + beta * env_le(sc, sc.lights[sc.infinite_lights[k]], d);
      P.L[p] = make_float4(l.r, l.g, l.b, 0.f);
    }
  }
}

// ---- connect_resolve ---------------------------------------------------------------------------------
// Second half of estimate_direct at full warp width, in connect-queue order: Ld_light (unoccluded shadow
// segment, integrator.rs:66-80) + Ld_bsdf (emitted radiance found by the MIS ray, integrator.rs:113-135), then
// L += beta * n_lights * Ld (integrator.rs:443-447, uniform_sample_one_light :216).  One thread per record =
// one writer per path, so the per-path summation order is the reference's.
#define PT_RESOLVE_MIN_BLOCKS 4  // 64 registers, no spills: 32 warps per SM for what is a streaming pass with a rare heavy branch
__global__ void __launch_bounds__(256, PT_RESOLVE_MIN_BLOCKS) connect_resolve_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ PathArrays P, const int* __restrict__ q_nee, RoundCounters* ctr) {
  const uint32_t n = ctr->n_nee;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const NeeRec* rec = P.nee + i;
    const float4 n3 = rec->n3;
    const uint32_t nf = __float_as_uint(n3.w);
    const NeeRes res = ld256(P.nee_res + i);
    Spec ld = sp(0.0f);
    if ((nf & PT_NEE_SHADOW) && !res.occluded) ld = ld + sp(rec->n0.w, rec->n1.w, rec->n2.w);
    const float4 n5 = rec->n5;
    if (nf & PT_NEE_MIS) {
      const int light_idx = (int)(nf & PT_NEE_LIGHT_MASK);
      const V3 md = mk3(n3);
      Spec li = sp(0.0f);
      if (res.prim >= 0) {
        const int hl = __float_as_int(__ldg(&sc.tri_verts[3 * (size_t)res.prim + 1].w));
        if (hl == light_idx) {
          SurfInter si;
          reconstruct_hit(sc, res.prim, res.b0, res.b1, res.b2, md, &si);
          li = area_le(sc, hl, si, -md);
        }
      } else if (sc.lights[light_idx].type == PTRS_LIGHT_INFINITE) {
        li = env_le(sc, sc.lights[light_idx], md);
      }
      if (!is_black(li)) {
        const float4 n4 = rec->n4;
        ld = ld + sp(n4.x, n4.y, n4.z) * li * sp(1.0f) * n4.w / n5.w;
      }
    }
    const int p = q_nee[i];
    const float4 l4 = P.L[p];
    const Spec L = sp(l4.x, l4.y, l4.z) + sp(n5.x, n5.y, n5.z) * ((float)sc.n_lights * ld);
    P.L[p] = make_float4(L.r, L.g, L.b, 0.f);
  }
}

// ---- accumulate ------------------------------------------------------------------------------------
// FilmTile::add_sample + merge_film_tile (film.rs:60-106, 213-228) straight into the film with
// 128-bit float atomics (red.global.add.v4.f32, sm_90+).
__global__ void __launch_bounds__(256) accumulate_kernel(const __grid_constant__ RenderConst rc, PathArrays P, uint32_t n, float4* film) {
  const uint32_t stride = gridDim.x * blockDim.x;
  const int W = rc.cam.width, H = rc.cam.height;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float2 pf = *reinterpret_cast<const float2*>(&P.slot[i].a.fx);
    if (pf.x < -1e29f) continue;
    const float4 l = P.L[i];
    const float dx = pf.x - 0.5f, dy = pf.y - 0.5f;
    int p0x = (int)ceilf(dx - rc.filter_radius[0]), p0y = (int)ceilf(dy - rc.filter_radius[1]);
    int p1x = (int)(floorf(dx + rc.filter_radius[0]) + 1.0f), p1y = (int)(floorf(dy + rc.filter_radius[1]) + 1.0f);
    p0x = max(p0x, 0);
    p0y = max(p0y, 0);
    p1x = min(p1x, W);
    p1y = min(p1y, H);
    for (int y = p0y; y < p1y; ++y) {
      const float fy = fabsf(((float)y - dy) * rc.inv_filter_radius[1] * 16.0f);
      const int iy = min((int)floorf(fy), 15);
      for (int x = p0x; x < p1x; ++x) {
        const float fx = fabsf(((float)x - dx) * rc.inv_filter_radius[0] * 16.0f);
        const int ix = min((int)floorf(fx), 15);
        const float w = rc.filter_table[iy * 16 + ix];
        atomicAdd(&film[(size_t)y * W + x], make_float4(l.x * w, l.y * w, l.z * w, w));
      }
    }
  }
}

// ---- read-bandwidth probe -------------------------------------------------------------------------------
// The denominator for "fraction of the L2 roofline" (SURVEY.md §8d: MEASURED_PEAKS.json holds no L2 figure): every
// thread streams 256-bit non-coherent loads over a buffer `reps` times.  With a buffer that fits in L2 the passes after
// the first are served by L2; with one far larger than L2 the figure is the HBM read bandwidth.
__global__ void __launch_bounds__(256) read_probe_kernel(const float4* __restrict__ buf, size_t n_pairs, int reps, uint32_t* sink) {
  float acc = 0.f;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (int r = 0; r < reps; ++r)  // blocks rotate over the buffer from pass to pass, so no SM re-reads what its own L1 holds
    for (size_t i = ((blockIdx.x + (size_t)r * 61u) % gridDim.x) * (size_t)blockDim.x + threadIdx.x; i < n_pairs; i += stride) {
      float a, b, c, d, e, f, g, h;
      asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                   : "=f"(a), "=f"(b), "=f"(c), "=f"(d), "=f"(e), "=f"(f), "=f"(g), "=f"(h)
                   : "l"(buf + 2 * i));
      acc += a + b + c + d + e + f + g + h;
    }
  if (acc == 123.456f) *sink = 1u;  // keeps the loads alive
}
// The traversal's own access pattern: independent 64-byte gathers (one sibling pair = two 32-byte records) at
// pseudo-random 64-byte-aligned positions, as many in flight as the hardware takes.  What a node fetch stream can
// reach at best from L2 (buffer <= L2) or from HBM (buffer >> L2).
__global__ void __launch_bounds__(256) gather_probe_kernel(const float4* __restrict__ buf, size_t n_blocks64, int per_thread, uint32_t* sink) {
  float acc = 0.f;
  uint64_t x = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull;
  for (int k = 0; k < per_thread; ++k) {
    x ^= x >> 30;  // splitmix64 step: independent of the loaded data, so gathers overlap
    x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27;
    x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    const float4* p = buf + 4 * (size_t)(x % n_blocks64);
    float a, b, c, d, e, f, g, h, a2, b2, c2, d2, e2, f2, g2, h2;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d), "=f"(e), "=f"(f), "=f"(g), "=f"(h) : "l"(p));
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a2), "=f"(b2), "=f"(c2), "=f"(d2), "=f"(e2), "=f"(f2), "=f"(g2), "=f"(h2)
                 : "l"(p + 2));
    acc += a + b + c + d + e + f + g + h + a2 + b2 + c2 + d2 + e2 + f2 + g2 + h2;
  }
  if (acc == 123.456f) *sink = 1u;
}
void launch_gather_probe(cudaStream_t st, int sm, const float4* buf, size_t n_blocks64, int per_thread, uint32_t* sink, uint64_t* n_gathers) {
  const int grid = PT_GRID(gather_probe_kernel, 256, sm);
  *n_gathers = (uint64_t)grid * 256u * (uint64_t)per_thread;
  gather_probe_kernel<<<grid, 256, 0, st>>>(buf, n_blocks64, per_thread, sink);
}
void launch_read_probe(cudaStream_t st, int sm, const float4* buf, size_t n_pairs, int reps, uint32_t* sink) {
  const int grid = PT_GRID(read_probe_kernel, 256, sm);
  read_probe_kernel<<<grid, 256, 0, st>>>(buf, n_pairs, reps, sink);
}

// ---- Distribution1D guide tables ----------------------------------------------------------------------
// guide[row][k] = #{ i < size : cdf[row][i] <= k / K }, k = 0..K (see DevEnv)
__global__ void build_guide_kernel(const float* __restrict__ cdf, uint32_t size, uint32_t rows, uint32_t K, uint32_t* __restrict__ guide) {
  const uint64_t total = (uint64_t)rows * (K + 1);
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t row = (uint32_t)(t / (K + 1)), k = (uint32_t)(t % (K + 1));
    const float* c = cdf + (size_t)row * size;
    const float u = (float)k / (float)K;
    uint32_t first = 0, len = size;
    while (len > 0) {
      const uint32_t half = len >> 1, middle = first + half;
      if (c[middle] <= u) {
        first = middle + 1;
        len -= half + 1;
      } else {
        len = half;
      }
    }
    guide[t] = first;
  }
}
void launch_build_guide(cudaStream_t st, const float* cdf, uint32_t size, uint32_t rows, uint32_t K, uint32_t* guide) {
  const uint64_t total = (uint64_t)rows * (K + 1);
  const int grid = (int)std::min<uint64_t>((total + 255) / 256, 148 * 16);
  build_guide_kernel<<<grid, 256, 0, st>>>(cdf, size, rows, K, guide);
}

// ---- parity probes -----------------------------------------------------------------------------------
// generic != 0: every draw through sobol_interval_to_index + sobol_sample (the reference's two functions);
// generic == 0: through the split tables, as the render kernels draw
__global__ void sobol_probe_kernel(const __grid_constant__ RenderConst rc, const uint32_t* __restrict__ sobol, const int* xy, const int* s,
                                   uint32_t n, const int* dims, uint32_t n_dims, float* out, uint64_t* out_index, int generic) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  PathSampler ps;
  sampler_start(rc.sobol, rc.split, ps, xy[2 * i], xy[2 * i + 1], (uint32_t)s[i], 0u);
  if (out_index) out_index[i] = sobol_interval_to_index(rc.sobol, (uint64_t)s[i], ps.px - rc.sobol.bounds_min[0], ps.py - rc.sobol.bounds_min[1]);
  SobolSplit sp = rc.split;
  if (generic) sp.stride = 0u;
  for (uint32_t k = 0; k < n_dims; ++k) out[(size_t)i * n_dims + k] = sample_dimension(rc.sobol, sp, sobol, ps, (uint32_t)dims[k]);
}

// ---- Sobol split tables (dev_sobol.cuh) ---------------------------------------------------------------
// row r < row_x: sample number r at pixel offset (0, 0); row_x <= r < row_y: pixel-x offset r - row_x, sample 0;
// r >= row_y: pixel-y offset.  Each entry = sobol_raw(sobol_interval_to_index(...), d), the reference's functions.
__global__ void sobol_split_build_kernel(const __grid_constant__ RenderConst rc, const uint32_t* __restrict__ sobol, uint32_t* __restrict__ tab) {
  const SobolSplit& sp = rc.split;
  const uint64_t total = (uint64_t)sp.n_rows * sp.stride;
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t r = (uint32_t)(t / sp.stride), d = (uint32_t)(t % sp.stride);
    uint64_t frame = 0;
    int32_t x = 0, y = 0;
    if (r < sp.row_x) frame = r;
    else if (r < sp.row_y) x = (int32_t)(r - sp.row_x);
    else y = (int32_t)(r - sp.row_y);
    tab[t] = sobol_raw(sobol, sobol_interval_to_index(rc.sobol, frame, x, y), d);
  }
}
void launch_sobol_split_build(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, uint32_t* tab) {
  const uint64_t total = (uint64_t)rc.split.n_rows * rc.split.stride;
  const int grid = (int)std::min<uint64_t>((total + 255) / 256, 148 * 8);
  sobol_split_build_kernel<<<grid, 256, 0, st>>>(rc, sobol, tab);
}

__global__ void ray_probe_kernel(const __grid_constant__ RenderConst rc, const uint32_t* __restrict__ sobol, const int* xy, const int* s,
                                 uint32_t n, PtrsRay* rays, float* p_film, float* rxry) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  PathSampler ps;
  sampler_start(rc.sobol, rc.split, ps, xy[2 * i], xy[2 * i + 1], (uint32_t)s[i], 0u);
  V2 u = get_2d(rc.sobol, rc.split, sobol, ps);
  const float fx = (float)ps.px + u.x, fy = (float)ps.py + u.y;
  V3 o, d, rx, ry;
  camera_ray(rc.cam, fx, fy, rc.diff_scale, &o, &d, &rx, &ry);
  rays[i].o[0] = o.x; rays[i].o[1] = o.y; rays[i].o[2] = o.z;
  rays[i].d[0] = d.x; rays[i].d[1] = d.y; rays[i].d[2] = d.z;
  rays[i].t_max = CUDART_INF_F;
  if (p_film) { p_film[2 * i] = fx; p_film[2 * i + 1] = fy; }
  if (rxry) {
    rxry[6 * i] = rx.x; rxry[6 * i + 1] = rx.y; rxry[6 * i + 2] = rx.z;
    rxry[6 * i + 3] = ry.x; rxry[6 * i + 4] = ry.y; rxry[6 * i + 5] = ry.z;
  }
}

// Film::to_channel_updates (film.rs:253-271) and to_rgba_image (film.rs:230-251, spectrum.rs:95-102)
__global__ void resolve_kernel(const float4* film, uint32_t n, float* rgb, uint8_t* rgba8) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = film[i];
  const float inv_wt = 1.f / p.w;
  const float c[3] = {p.x * inv_wt, p.y * inv_wt, p.z * inv_wt};
  if (rgb) {
    rgb[3 * i] = c[0];
    rgb[3 * i + 1] = c[1];
    rgb[3 * i + 2] = c[2];
  }
  if (rgba8) {
    for (int k = 0; k < 3; ++k) {
      float v = c[k];
      float gc = v <= 0.0031308f ? 12.92f * v : 1.055f * powf(v, 1.0f / 2.4f) - 0.055f;  // math.rs:133-139
      float q = rclamp(gc * 255.0f + 0.5f, 0.0f, 255.0f);
      rgba8[4 * i + k] = (uint8_t)q;  // NaN -> 0 like Rust's saturating cast
    }
    rgba8[4 * i + 3] = 255;
  }
}


// ---- launchers -----------------------------------------------------------------------------------------
void launch_generate(cudaStream_t st, int sm, const RenderConst& rc, const uint32_t* sobol, const PathArrays& P, uint64_t work_base,
                     uint32_t n_work, const int* list_xy, const int* list_s, int* q_ext, RoundCounters* ctr) {
  const int grid = PT_GRID(generate_kernel, 256, sm);
  generate_kernel<<<grid, 256, 0, st>>>(rc, sobol, P, work_base, n_work, list_xy, list_s, q_ext, ctr);
}
void launch_shade_miss(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, const int* q, RoundCounters* ctr) {
  const int grid = PT_GRID(shade_miss_kernel, 128, sm);
  shade_miss_kernel<<<grid, 128, 0, st>>>(sc, P, q, ctr);
}
void launch_connect_resolve(cudaStream_t st, int sm, const DevScene& sc, const PathArrays& P, const int* q_nee, RoundCounters* ctr) {
  const int grid = PT_GRID(connect_resolve_kernel, 256, sm);
  connect_resolve_kernel<<<grid, 256, 0, st>>>(sc, P, q_nee, ctr);
}
void launch_accumulate(cudaStream_t st, int sm, const RenderConst& rc, const PathArrays& P, uint32_t n, float4* film) {
  const int grid = PT_GRID(accumulate_kernel, 256, sm);
  accumulate_kernel<<<grid, 256, 0, st>>>(rc, P, n, film);
}
void launch_resolve(cudaStream_t st, const float4* film, uint32_t n, float* rgb, uint8_t* rgba8) {
  resolve_kernel<<<(n + 255) / 256, 256, 0, st>>>(film, n, rgb, rgba8);
}
void launch_sobol_probe(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, const int* xy, const int* s, uint32_t n,
                        const int* dims, uint32_t n_dims, float* out, uint64_t* out_index, int generic) {
  sobol_probe_kernel<<<(n + 127) / 128, 128, 0, st>>>(rc, sobol, xy, s, n, dims, n_dims, out, out_index, generic);
}
void launch_ray_probe(cudaStream_t st, const RenderConst& rc, const uint32_t* sobol, const int* xy, const int* s, uint32_t n, PtrsRay* rays,
                      float* p_film, float* rxry) {
  ray_probe_kernel<<<(n + 127) / 128, 128, 0, st>>>(rc, sobol, xy, s, n, rays, p_film, rxry);
}

}  // namespace ptrs
