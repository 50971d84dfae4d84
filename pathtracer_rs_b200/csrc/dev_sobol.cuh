// Global Sobol sampler on the device: src/pathtracer/sampler/sobol.rs:81-193,
// src/pathtracer/lowdiscrepancy.rs:9-57.  Integer XOR networks; bit-exact with the CPU path.
#pragma once
#include "dev_math.cuh"

namespace ptrs {

// VD_C_SOBOL_MATRICES[m-1] / VD_C_SOBOL_MATRICES_INV[m-1] for the render's log2 resolution m
// (at most 52 u64 each), uploaded per render into constant memory.
struct SobolConfig {
  uint64_t vdc[52];
  uint64_t vdc_inv[52];
  int32_t bounds_min[2];
  int32_t resolution;
  uint32_t log2_resolution;
  uint32_t n_vdc, n_vdc_inv;
  int32_t spp;  // rounded up to a power of two
  int32_t pad;
};

#define PT_SOBOL_COLS 52
#define PT_ARRAY_START_DIM 5

// lowdiscrepancy.rs:9-39
PT_DEV uint64_t sobol_interval_to_index(const SobolConfig& c, uint64_t frame, int32_t px, int32_t py) {
  const uint32_t m = c.log2_resolution;
  if (m == 0) return 0;
  uint64_t index = frame << (m << 1);
  uint64_t delta = 0;
  for (int k = 0; frame != 0; frame >>= 1, ++k)
    if (frame & 1) delta ^= c.vdc[k];
  uint64_t b = ((uint64_t)(((uint32_t)px) << m) | (uint64_t)(int64_t)py) ^ delta;
  for (int k = 0; b != 0; b >>= 1, ++k)
    if (b & 1) index ^= c.vdc_inv[k];
  return index;
}

// lowdiscrepancy.rs:42-57
PT_DEV float sobol_sample(const uint32_t* __restrict__ matrices, uint64_t index, uint32_t dimension, uint32_t scramble) {
  uint32_t v = scramble;
  const uint32_t* col = matrices + dimension * PT_SOBOL_COLS;
  uint32_t lo = (uint32_t)index, hi = (uint32_t)(index >> 32);
  while (lo) {
    int k = __ffs(lo) - 1;
    v ^= __ldg(col + k);
    lo &= lo - 1;
  }
  while (hi) {
    int k = __ffs(hi) - 1;
    v ^= __ldg(col + 32 + k);
    hi &= hi - 1;
  }
  return fminf(PT_ONE_MINUS_EPSILON, (float)v * 0x1.p-32f);
}

// ---- split tables ------------------------------------------------------------------------------------
// Both steps of a draw are linear maps over GF(2): sobol_interval_to_index() XORs one column per set bit of
// `frame` and of ((px << m) | py) ^ delta(frame), and sobol_sample() XORs one matrix column per set bit of
// the index.  With px, py < 2^m the three inputs occupy disjoint bits, so
//     raw(sample s, pixel (px, py), dimension d) = S_d[s] ^ X_d[px] ^ Y_d[py] ^ scramble
// where each table entry is the reference's own pair of functions evaluated with the other two inputs
// zero.  sobol_split_build_kernel fills the tables with exactly those functions once per render setup
// (rows: spp samples, then x extent, then y extent; `stride` dimensions per row), and a draw in the shade
// kernels is three 4-byte loads and three XORs instead of a loop over the ~28 set bits of the index.
// Values are bit-identical to sobol_sample() (tests/test_gpu_parity.py::test_sobol_*).
struct SobolSplit {
  const uint32_t* tab;
  uint32_t stride;        // dimensions per row (multiple of 4); draws at dimension >= stride take the generic path
  uint32_t row_x, row_y;  // first row of the pixel-x / pixel-y blocks (sample rows start at 0)
  uint32_t n_rows;
};

// the u32 before scrambling and scaling (lowdiscrepancy.rs:45-55 without `v = scramble`)
PT_DEV uint32_t sobol_raw(const uint32_t* __restrict__ matrices, uint64_t index, uint32_t dimension) {
  uint32_t v = 0;
  const uint32_t* col = matrices + dimension * PT_SOBOL_COLS;
  for (int k = 0; index != 0; index >>= 1, ++k)
    if (index & 1) v ^= __ldg(col + k);
  return v;
}

// Per-path sampler state: the reference's SobolSampler minus everything that is constant per render.
struct PathSampler {
  uint32_t scramble;  // current_scramble_index as u32
  uint32_t dimension;
  int32_t px, py;
  uint32_t sample;               // sample number of the pixel (the `frame` of sobol_interval_to_index)
  uint32_t row_s, row_x, row_y;  // element offsets of this path's three rows in SobolSplit::tab
};

PT_DEV uint32_t pixel_scramble(int32_t x, int32_t y) {  // sobol.rs:83-86 (+ `scramble as u32`)
  return (uint32_t)cantor_pairing((uint64_t)(int64_t)(x + PT_HALF_MAX_I32), (uint64_t)(int64_t)(y + PT_HALF_MAX_I32));
}

PT_DEV void sampler_start(const SobolConfig& c, const SobolSplit& sp, PathSampler& s, int32_t px, int32_t py, uint32_t sample, uint32_t dimension) {
  s.px = px;
  s.py = py;
  s.sample = sample;
  s.dimension = dimension;
  s.scramble = pixel_scramble(px, py);
  s.row_s = sample * sp.stride;
  s.row_x = (sp.row_x + (uint32_t)(px - c.bounds_min[0])) * sp.stride;
  s.row_y = (sp.row_y + (uint32_t)(py - c.bounds_min[1])) * sp.stride;
}

// generic path (sobol.rs:169-193): only reached for dimensions beyond the split tables
// (the sampler's fields by value: a reference would keep the caller's PathSampler in local memory)
PT_DEVN float sample_dimension_generic(const SobolConfig& c, const uint32_t* __restrict__ matrices, uint32_t sample, int32_t px, int32_t py,
                                       uint32_t scramble, uint32_t dim) {
  const uint64_t index = sobol_interval_to_index(c, (uint64_t)sample, px - c.bounds_min[0], py - c.bounds_min[1]);
  return sobol_sample(matrices, index, dim, scramble);
}

PT_DEV float sample_dimension(const SobolConfig& c, const SobolSplit& sp, const uint32_t* __restrict__ matrices, const PathSampler& s, uint32_t dim) {
  float v;
  if (dim < sp.stride) {
    const uint32_t raw = __ldg(sp.tab + s.row_s + dim) ^ __ldg(sp.tab + s.row_x + dim) ^ __ldg(sp.tab + s.row_y + dim) ^ s.scramble;
    v = fminf(PT_ONE_MINUS_EPSILON, (float)raw * 0x1.p-32f);
  } else {
    v = sample_dimension_generic(c, matrices, s.sample, s.px, s.py, s.scramble, dim);
  }
  if (dim == 0 || dim == 1) {
    int32_t pmin = dim == 0 ? c.bounds_min[0] : c.bounds_min[1];
    int32_t pix = dim == 0 ? s.px : s.py;
    v = v * (float)c.resolution + (float)pmin;
    v = rclamp(v - (float)pix, 0.f, PT_ONE_MINUS_EPSILON);
  }
  return v;
}
PT_DEV float get_1d(const SobolConfig& c, const SobolSplit& sp, const uint32_t* __restrict__ m, PathSampler& s) {  // sobol.rs:129-137 (array range empty)
  float v = sample_dimension(c, sp, m, s, s.dimension);
  s.dimension += 1;
  return v;
}
PT_DEV V2 get_2d(const SobolConfig& c, const SobolSplit& sp, const uint32_t* __restrict__ m, PathSampler& s) {  // sobol.rs:139-151
  if (s.dimension + 1 >= PT_ARRAY_START_DIM && s.dimension < PT_ARRAY_START_DIM) s.dimension = PT_ARRAY_START_DIM;
  V2 v{sample_dimension(c, sp, m, s, s.dimension), sample_dimension(c, sp, m, s, s.dimension + 1)};
  s.dimension += 2;
  return v;
}

}  // namespace ptrs
