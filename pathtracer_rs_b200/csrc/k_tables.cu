// Table construction on the device (SURVEY.md §8f-2): what the reference's importers build on the host right
// before the path runs —
//   MIPMap::new's box-filtered pyramid                     src/pathtracer/texture.rs:345-405
//   InfiniteAreaLight::new's sampling density              src/pathtracer/light.rs:372-387
//   Distribution1D::new / Distribution2D::new              src/pathtracer/sampling.rs:133-162, 185-209
// — as kernels, so that a scene description may carry level 0 of an image only and no Distribution2D arrays (for
// the 1k environment map of BASELINE configs[1] that is 10.7 MB less pyramid and 16.8 MB less distribution to
// assemble on the host and to copy).  Built with the exact units' flags (no FMA contraction, IEEE division): every
// value is bit-identical to host/scene_builder.cpp's, which is what tests/test_gpu_parity.py checks.  The two places
// where the host path goes through libm — sin(pi v) per row of the density and log2 of the filter width — are
// evaluated by the library's host code and handed to the kernels, so they are the same glibc values.
#include <algorithm>

#include "launch.hpp"
#include "wavefront.cuh"

namespace ptrs {

namespace {

// level i from level i - 1: mean of the 2 x 2 block, addressed through the wrap mode (texture.rs:386-402)
__global__ void __launch_bounds__(256) mip_level_kernel(const float* __restrict__ prev, int pw, int ph, int channels, int wrap, float* __restrict__ out, int sres,
                                                        int tres) {
  const uint32_t n = (uint32_t)sres * (uint32_t)tres;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int s = (int)(i % (uint32_t)sres), t = (int)(i / (uint32_t)sres);
    auto texel = [&](int ss, int tt, int c) -> float {
      if (wrap == PTRS_WRAP_REPEAT) {
        ss = abs_mod(ss, pw);
        tt = abs_mod(tt, ph);
      } else if (wrap == PTRS_WRAP_BLACK) {
        if (ss < 0 || ss >= pw || tt < 0 || tt >= ph) return 0.f;
      } else {
        ss = min(max(ss, 0), pw - 1);
        tt = min(max(tt, 0), ph - 1);
      }
      return prev[((size_t)tt * pw + ss) * channels + c];
    };
    for (int c = 0; c < channels; ++c)
      out[(size_t)i * channels + c] = (((texel(2 * s, 2 * t, c) + texel(2 * s + 1, 2 * t, c)) + texel(2 * s, 2 * t + 1, c)) + texel(2 * s + 1, 2 * t + 1, c)) * 0.25f;
  }
}

// func[v][u] = sin(pi (v + 0.5) / nv) * y(MIPMap::lookup_width((u + 0.5) / nu, (v + 0.5) / nv, filter width))   light.rs:375-387
// mode: 0 = finest level only, 1 = coarsest level only, 2 = lerp(level il, il + 1, delta)   (texture.rs:447-464)
__global__ void __launch_bounds__(256) env_density_kernel(const __grid_constant__ DevScene sc, int mip, int nu, int nv, const float* __restrict__ row_sin, int mode,
                                                          int il, float delta, float* __restrict__ func) {
  const PtrsMipMap& mm = sc.mipmaps[mip];
  const uint32_t n = (uint32_t)nu * (uint32_t)nv;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int u = (int)(i % (uint32_t)nu), v = (int)(i / (uint32_t)nu);
    const float up = ((float)u + 0.5f) / (float)nu, vp = ((float)v + 0.5f) / (float)nv;
    Spec c;
    if (mode == 0) {
      c = mip_triangle(sc, mm, 0, up, vp);
    } else if (mode == 1) {
      c = mip_triangle(sc, mm, mm.n_levels - 1, up, vp);
    } else {
      const Spec a = mip_triangle(sc, mm, il, up, vp), b = mip_triangle(sc, mm, il + 1, up, vp);
      c = sp(a.r * (1.0f - delta) + b.r * delta, a.g * (1.0f - delta) + b.g * delta, a.b * (1.0f - delta) + b.b * delta);
    }
    const float y = c.r * 0.212671f + c.g * 0.715160f + c.b * 0.072169f;  // spectrum.rs:112-115
    func[i] = row_sin[v] * y;
  }
}

// Distribution1D::new for `rows` independent rows of n entries.  The running sum is sequential in the reference
// (sampling.rs:139-145) and float addition does not associate, so ONE thread walks a row from left to right — but the
// row is brought to it through shared memory in 32 x 32 tiles loaded and stored with coalesced accesses (a thread per
// row reading its row straight from global memory touches a 32-byte sector per 4-byte entry: 1.5 ms for the 2048 x 1024
// table of the 1k map, against ~0.1 ms this way).  cdf: rows x (n + 1); func_int: rows.
__global__ void __launch_bounds__(256) row_prefix_kernel(const float* __restrict__ func, int n, int rows, float* __restrict__ cdf, float* __restrict__ func_int) {
  __shared__ float tile[32][33];
  const int row0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float acc = 0.f;  // threads 0 .. 31: thread t carries the running sum of row row0 + t
  for (int col0 = 0; col0 < n; col0 += 32) {
    for (int r = ty; r < 32; r += 8) {
      const int row = row0 + r, col = col0 + tx;
      tile[r][tx] = (row < rows && col < n) ? func[(size_t)row * n + col] : 0.f;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      const int r = threadIdx.x;
      for (int c = 0; c < 32; ++c)
        if (col0 + c < n) {
          acc = acc + tile[r][c] / (float)n;
          tile[r][c] = acc;
        }
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
      const int row = row0 + r, col = col0 + tx;
      if (row < rows && col < n) cdf[(size_t)row * (n + 1) + 1 + col] = tile[r][tx];
    }
    __syncthreads();
  }
  if (threadIdx.x < 32 && row0 + (int)threadIdx.x < rows) {
    func_int[row0 + threadIdx.x] = acc;
    cdf[(size_t)(row0 + threadIdx.x) * (n + 1)] = 0.f;
  }
}
// second half of Distribution1D::new (sampling.rs:146-156): cdf[i] /= func_int, or i / n when the row integrates to zero
__global__ void __launch_bounds__(256) row_normalise_kernel(int n, int rows, float* __restrict__ cdf, const float* __restrict__ func_int) {
  const size_t total = (size_t)rows * (n + 1);
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int row = (int)(t / (size_t)(n + 1)), i = (int)(t % (size_t)(n + 1));
    if (i == 0) continue;
    const float fi = func_int[row];
    cdf[t] = fi == 0.0f ? (float)i / (float)n : cdf[t] / fi;
  }
}

// per-triangle shading record (dev_scene.cuh tri_shade)
__global__ void __launch_bounds__(256) pack_shading_kernel(uint32_t n, const float4* __restrict__ tri_verts, const uint4* __restrict__ tri_index,
                                                           const float* __restrict__ normal, const float* __restrict__ uv, float4* __restrict__ out) {
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const uint32_t flags = __float_as_uint(tri_verts[3 * (size_t)k + 2].w) & 0xffu;
    const uint4 idx = tri_index[k];
    const uint32_t v[3] = {idx.x, idx.y, idx.z};
    float r[16];
    for (int j = 0; j < 16; ++j) r[j] = 0.f;
    if ((flags & PTRS_MESH_HAS_NORMAL) && normal)
      for (int j = 0; j < 3; ++j)
        for (int c = 0; c < 3; ++c) r[3 * j + c] = normal[3 * (size_t)v[j] + c];
    if ((flags & PTRS_MESH_HAS_UV) && uv) {
      for (int j = 0; j < 3; ++j)
        for (int c = 0; c < 2; ++c) r[9 + 2 * j + c] = uv[2 * (size_t)v[j] + c];
    } else {  // shape.rs:34-48
      r[9] = 0.f, r[10] = 0.f, r[11] = 1.f, r[12] = 0.f, r[13] = 1.f, r[14] = 1.f;
    }
    for (int j = 0; j < 4; ++j) out[4 * (size_t)k + j] = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
  }
}

}  // namespace

void launch_pack_shading(cudaStream_t st, uint32_t n, const float4* tri_verts, const uint4* tri_index, const float* normal, const float* uv, float4* out) {
  if (n == 0) return;
  const int grid = (int)std::min<uint32_t>((n + 255u) / 256u, 148u * 8u);
  pack_shading_kernel<<<grid, 256, 0, st>>>(n, tri_verts, tri_index, normal, uv, out);
}
void launch_mip_level(cudaStream_t st, const float* prev, int pw, int ph, int channels, int wrap, float* out, int sres, int tres) {
  const uint32_t n = (uint32_t)sres * (uint32_t)tres;
  const int grid = (int)std::min<uint32_t>((n + 255u) / 256u, 148u * 8u);
  mip_level_kernel<<<grid, 256, 0, st>>>(prev, pw, ph, channels, wrap, out, sres, tres);
}
void launch_env_density(cudaStream_t st, const DevScene& sc, int mip, int nu, int nv, const float* row_sin, int mode, int il, float delta, float* func) {
  const uint32_t n = (uint32_t)nu * (uint32_t)nv;
  const int grid = (int)std::min<uint32_t>((n + 255u) / 256u, 148u * 16u);
  env_density_kernel<<<grid, 256, 0, st>>>(sc, mip, nu, nv, row_sin, mode, il, delta, func);
}
void launch_row_cdf(cudaStream_t st, const float* func, int n, int rows, float* cdf, float* func_int) {
  row_prefix_kernel<<<(rows + 31) / 32, 256, 0, st>>>(func, n, rows, cdf, func_int);
  const size_t total = (size_t)rows * (n + 1);
  const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  row_normalise_kernel<<<grid, 256, 0, st>>>(n, rows, cdf, func_int);
}

}  // namespace ptrs
