// Whole-scene inference around the generator: cut overlapping windows of a scene into the generator's NCHW fp32 batch
// layout, and blend the per-tile predictions back into one NIR band.  The reference only runs pre-cut tiles
// (create_synthetic_dataset.py:93,100-118); these kernels replace the per-tile `model(hr)` loop's hand-written
// cutting and stitching.  All are HBM-bound single passes; none uses atomics, so results are bit-reproducible.
//
// Nodata (GDAL's per-dataset mask): a pixel is nodata when every channel equals the nodata value (NaN matches NaN).
// ng_scene_tile_valid counts the valid pixels of each window so that the host can skip windows without one;
// ng_scene_blend_masked blends a compacted prediction buffer and writes nodata pixels as a fill value.
//
// Index bands: ng_scene_blend_indices also writes, after the NIR plane, index-mode RemoteSensingIndices planes (epsilon
// 0, the formulas of rs_index.cuh that ng_rs_index evaluates) of each pixel's blended NIR and its R, G, B (channels 0-2
// of the resident scene rows, converted as ng_scene_tiles converts them); nodata pixels are the fill value in every plane.
//
// Blend (nirgan_b200/scene.py states the same definitions):
//   out(y, x) = sum_t w_t(y, x) p_t(y, x) / sum_t w_t(y, x)   over the tiles t covering (y, x), ascending (k_y, k_x)
//   w(i, j)   = w1(i) w1(j),   w1(i) = min(i + 1, T - i, overlap + 1) / (overlap + 1)
// computed with the integer weights (overlap + 1)^2 w(i, j), and a pixel covered by a single tile takes that tile's value unchanged.
#include "common.cuh"
#include "rs_index.cuh"

namespace ng {

constexpr int SC_THREADS = 256;

template <typename E> __device__ __forceinline__ float scene_value(E v, float dn_scale);
template <> __device__ __forceinline__ float scene_value<float>(float v, float) { return v; }
// IEEE division (the library is built without fast math): bit-identical to torch's `scene.float() / dn_scale`
template <> __device__ __forceinline__ float scene_value<uint16_t>(uint16_t v, float dn_scale) {
  return __fdiv_rn((float)v, dn_scale);
}

// one block row per (tile, channel); V consecutive elements of a tile row per thread (V = 4 when T % 4 == 0: one
// 16-byte store).  A window outside the resident rows is written as NaN instead of being read out of bounds.
template <typename E, int V>
__global__ void __launch_bounds__(SC_THREADS)
scene_tiles_kernel(const E* __restrict__ scene, int C, int rows, int W, int row0, const int2* __restrict__ origins,
                   int T, float dn_scale, float* __restrict__ dst) {
  const int tile = blockIdx.z, c = blockIdx.y;
  const int2 o = origins[tile];                       // (y0, x0) in scene coordinates
  const int r = o.x - row0;
  const bool inside = r >= 0 && r + T <= rows && o.y >= 0 && o.y + T <= W;
  const E* src = scene + ((size_t)c * rows + (inside ? r : 0)) * W + (inside ? o.y : 0);
  float* d = dst + ((size_t)tile * C + c) * T * T;
  const int per_row = T / V, total = T * per_row;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int i = e / per_row, j = (e - i * per_row) * V;
    float v[V];
#pragma unroll
    for (int k = 0; k < V; ++k) v[k] = inside ? scene_value<E>(src[(size_t)i * W + j + k], dn_scale) : __int_as_float(0x7fc00000);
    if constexpr (V == 4) *reinterpret_cast<float4*>(d + (size_t)i * T + j) = make_float4(v[0], v[1], v[2], v[3]);
    else d[(size_t)i * T + j] = v[0];
  }
}

// v == nodata, with NaN matching NaN (so -0.0 matches 0.0); uint16 values are exact in fp32
template <typename E> __device__ __forceinline__ bool is_nodata(E v, float nodata);
template <> __device__ __forceinline__ bool is_nodata<float>(float v, float nodata) {
  return v == nodata || (v != v && nodata != nodata);
}
template <> __device__ __forceinline__ bool is_nodata<uint16_t>(uint16_t v, float nodata) { return (float)v == nodata; }

// pixel `at` of the planes scene[c * plane ..]: valid unless every channel is nodata.  All channels are read (no early
// exit), so the loads of a thread issue together and the bytes read are C per pixel whatever the data.
template <typename E>
__device__ __forceinline__ bool pixel_valid(const E* __restrict__ scene, int C, size_t plane, size_t at, float nodata) {
  bool valid = false;
  for (int c = 0; c < C; ++c) valid |= !is_nodata<E>(scene[(size_t)c * plane + at], nodata);
  return valid;
}

// one block per window (a host scene's launch covers one tile row, a few dozen windows: 512 threads keep more loads in
// flight per SM than 256).  The count is a fixed-order integer reduction (warp sums, then the block's warp partials).
constexpr int SV_THREADS = 512;

template <typename E>
__global__ void __launch_bounds__(SV_THREADS)
scene_valid_kernel(const E* __restrict__ scene, int C, int rows, int W, int row0, const int2* __restrict__ origins,
                   int T, float nodata, int* __restrict__ counts) {
  const int tile = blockIdx.x;
  const int2 o = origins[tile];                       // (y0, x0) in scene coordinates
  const int r = o.x - row0;
  if (!(r >= 0 && r + T <= rows && o.y >= 0 && o.y + T <= W)) {   // outside the resident rows: -1, nothing read
    if (threadIdx.x == 0) counts[tile] = -1;
    return;
  }
  const E* src = scene + (size_t)r * W + o.y;
  const size_t plane = (size_t)rows * W;
  int cnt = 0;
#pragma unroll 4
  for (int e = threadIdx.x; e < T * T; e += SV_THREADS) {
    const int i = e / T, j = e - i * T;
    cnt += pixel_valid<E>(src, C, plane, (size_t)i * W + j, nodata);
  }
  __shared__ int part[SV_THREADS / 32];
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x < 32) {
    cnt = __reduce_add_sync(0xffffffffu, threadIdx.x < SV_THREADS / 32 ? part[threadIdx.x] : 0);
    if (threadIdx.x == 0) counts[tile] = cnt;
  }
}

// the scene rows the blend reads (the nodata mask, the R, G, B of the index bands): scene rows [row0, row0 + rows)
// resident as scene [C][rows][W]
template <typename E> struct SceneMask {
  const E* scene;
  int C, rows, row0;
  float nodata, nodata_out;
};

// the index bands: which[0 .. k) in RS_TERMS numbering (1 = NDVI .. 6 = EVI), plane 1 + i is index which[i]
constexpr int SCENE_MAX_INDICES = 6;
struct SceneIndices {
  int which[SCENE_MAX_INDICES];
  int k;
  float dn_scale;
};

// index mode of RemoteSensingIndices (epsilon 0) at one pixel of NIR n: the prediction map of ng_rs_index
__device__ __forceinline__ float rs_index_value(int which, float n, float R, float G, float Bl) {
  switch (which) {
    case 1: return rs_ndvi(n, n, R, 0.f).ip;
    case 2: return rs_ndvi(n, n, G, 0.f).ip;
    case 3: return rs_gndvi(n, n, R, G).ip;
    case 4: return rs_savi(n, n, R).ip;
    case 5: return rs_msavi(n, n, R).ip;
    default: return rs_evi(n, n, R, Bl, 0.f).ip;
  }
}

template <int V> __device__ __forceinline__ void store_px(float* o, const float (&v)[V]) {
  if constexpr (V == 4) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
  else *o = v[0];
}

// (overlap + 1) * w1(i): the common factor cancels in the normalised sum, and the integer weights and their sums are
// exact in fp32 (at most (overlap + 1)^2 per tile)
__device__ __forceinline__ int blend_m1(int i, int T, int ov1) { return min(min(i + 1, T - i), ov1); }

// first index k of the ascending origins o[0..n) with o[k] + T > p (the first tile that can cover p)
__device__ __forceinline__ int first_cover(const int* __restrict__ o, int n, int T, int p) {
  int lo = 0, hi = n;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (o[mid] + T <= p) lo = mid + 1; else hi = mid; }
  return lo;
}

// out(y, x) over the covering tiles: rows ky0.. of oy, columns found here (ascending (ky, kx), fp32).  SLOT: tile
// ky * nx + kx is row slot[ky * nx + kx] of the compacted pred, and a skipped tile (-1) is passed over; it never covers
// a valid pixel, since a tile with a valid pixel is computed.  Without SLOT, tile ky * nx + kx is row ky * nx + kx.
template <bool SLOT>
__device__ __forceinline__ float blend_pixel(const float* __restrict__ pred, const int* __restrict__ slot,
                                             const int* __restrict__ oy, int ny, int ky0,
                                             const int* __restrict__ ox, int nx, int T, int ov1, int y, int x) {
  const int kx0 = first_cover(ox, nx, T, x);
  float acc = 0.f, wsum = 0.f, last = 0.f;
  int cnt = 0;
  for (int ky = ky0; ky < ny && oy[ky] <= y; ++ky) {
    const int i = y - oy[ky];
    const int my = blend_m1(i, T, ov1);
    const float* prow = pred + ((size_t)ky * nx) * T * T + (size_t)i * T;
    for (int kx = kx0; kx < nx && ox[kx] <= x; ++kx) {
      const int j = x - ox[kx];
      const float w = (float)(my * blend_m1(j, T, ov1));
      if constexpr (SLOT) {
        const int s = __ldg(slot + ky * nx + kx);
        if (s < 0) continue;
        last = __ldg(pred + (size_t)s * T * T + (size_t)i * T + j);
      } else {
        last = __ldg(prow + (size_t)kx * T * T + j);
      }
      acc = __fmaf_rn(w, last, acc);
      wsum = __fadd_rn(wsum, w);
      ++cnt;
    }
  }
  return cnt == 1 ? last : __fdiv_rn(acc, wsum);      // no covering tile: 0 / 0 = NaN marks the caller's error
}

// gather form: every output pixel of rows [y0, y0 + rows) reads its covering tiles and is written once.  V consecutive
// pixels of one row per thread (V = 4 when W % 4 == 0: one 16-byte store per plane).  SLOT: pred is compacted through
// slot.  MASK: a nodata pixel of the resident scene rows is written as mask.nodata_out without reading any prediction.
// INDEX: planes 1 .. idx.k (plane p at out + p * rows * W) get the index bands; the R, G, B loads serve the nodata test
// too.
template <int V, bool SLOT, bool MASK, bool INDEX, typename E = float>
__global__ void __launch_bounds__(SC_THREADS)
scene_blend_kernel(const float* __restrict__ pred, const int* __restrict__ slot, const int* __restrict__ oy, int ny,
                   const int* __restrict__ ox, int nx, int T, int overlap, int W, int y0, int rows, SceneMask<E> mask,
                   float* __restrict__ out, SceneIndices idx) {
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) * V;
  if (x >= W) return;
  const int ov1 = overlap + 1;
  for (int row = blockIdx.y; row < rows; row += gridDim.y) {
    const int y = y0 + row;
    const int ky0 = first_cover(oy, ny, T, y);
    float* o = out + (size_t)row * W + x;
    if constexpr (INDEX) {
      const size_t plane = (size_t)mask.rows * W;
      const E* s = mask.scene + (size_t)(y - mask.row0) * W + x;
      bool valid[V];
      float nir[V], R[V], G[V], Bl[V];
#pragma unroll
      for (int q = 0; q < V; ++q) {
        const E r = s[q], g = s[plane + q], b = s[2 * plane + q];
        valid[q] = true;
        if constexpr (MASK) {
          valid[q] = !is_nodata<E>(r, mask.nodata) | !is_nodata<E>(g, mask.nodata) | !is_nodata<E>(b, mask.nodata);
          for (int c = 3; c < mask.C; ++c) valid[q] |= !is_nodata<E>(s[(size_t)c * plane + q], mask.nodata);
        }
        nir[q] = valid[q] ? blend_pixel<SLOT>(pred, slot, oy, ny, ky0, ox, nx, T, ov1, y, x + q) : mask.nodata_out;
        R[q] = scene_value<E>(r, idx.dn_scale);
        G[q] = scene_value<E>(g, idx.dn_scale);
        Bl[q] = scene_value<E>(b, idx.dn_scale);
      }
      store_px<V>(o, nir);
      for (int p = 0; p < idx.k; ++p) {
        const int which = idx.which[p];
        float v[V];
#pragma unroll
        for (int q = 0; q < V; ++q)
          v[q] = valid[q] ? rs_index_value(which, nir[q], R[q], G[q], Bl[q]) : mask.nodata_out;
        store_px<V>(o + (size_t)(1 + p) * rows * W, v);
      }
    } else {
      auto px = [&](int xx) -> float {
        if constexpr (MASK) {
          const E* srow = mask.scene + (size_t)(y - mask.row0) * W;
          if (!pixel_valid<E>(srow, mask.C, (size_t)mask.rows * W, xx, mask.nodata)) return mask.nodata_out;
        }
        return blend_pixel<SLOT>(pred, slot, oy, ny, ky0, ox, nx, T, ov1, y, xx);
      };
      if constexpr (V == 4)
        *reinterpret_cast<float4*>(o) = make_float4(px(x), px(x + 1), px(x + 2), px(x + 3));
      else
        *o = px(x);
    }
  }
}

template <bool SLOT, bool MASK, bool INDEX, typename E>
int launch_blend(const float* pred, const int* slot, const int* oy, int ny, const int* ox, int nx, int T, int overlap,
                 int W, int y0, int y1, SceneMask<E> mask, SceneIndices idx, float* out, void* stream) {
  const bool vec = W % 4 == 0 && ((uintptr_t)out & 15) == 0;
  const int V = vec ? 4 : 1;
  const int per_row = (W + V - 1) / V;
  const dim3 grid((per_row + SC_THREADS - 1) / SC_THREADS, y1 - y0 < 65535 ? y1 - y0 : 65535);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec)
    scene_blend_kernel<4, SLOT, MASK, INDEX, E><<<grid, SC_THREADS, 0, st>>>(pred, slot, oy, ny, ox, nx, T, overlap, W,
                                                                             y0, y1 - y0, mask, out, idx);
  else
    scene_blend_kernel<1, SLOT, MASK, INDEX, E><<<grid, SC_THREADS, 0, st>>>(pred, slot, oy, ny, ox, nx, T, overlap, W,
                                                                             y0, y1 - y0, mask, out, idx);
  NG_LAUNCH_CHECK("scene_blend_kernel");
  return NG_OK;
}

// the four (SLOT, MASK) index blends of one element type
template <typename E>
int launch_blend_indices(const float* pred, const int* slot, const int* oy, int ny, const int* ox, int nx, int T,
                         int overlap, int W, int y0, int y1, SceneMask<E> sc, bool masked, SceneIndices idx,
                         float* out, void* stream) {
  if (slot)
    return masked ? launch_blend<true, true, true, E>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1, sc, idx, out, stream)
                  : launch_blend<true, false, true, E>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1, sc, idx, out, stream);
  return masked ? launch_blend<false, true, true, E>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1, sc, idx, out, stream)
                : launch_blend<false, false, true, E>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1, sc, idx, out, stream);
}

}  // namespace ng

using namespace ng;

extern "C" int ng_scene_tiles(const void* scene, int32_t dtype, int32_t C, int32_t rows, int32_t W, int32_t row0,
                              const int32_t* origins, int32_t n, int32_t T, float dn_scale, float* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(scene && origins && dst && C > 0 && rows > 0 && W > 0 && row0 >= 0 && n > 0 && T > 0, NG_E_ARG,
             "scene_tiles: bad arguments");
  NG_REQUIRE(dtype == NG_F32 || dtype == NG_U16, NG_E_ARG, "scene_tiles: the scene must be NG_F32 or NG_U16");
  NG_REQUIRE(dtype != NG_U16 || dn_scale > 0.f, NG_E_ARG, "scene_tiles: dn_scale must be positive");
  NG_REQUIRE(T <= rows && T <= W, NG_E_SHAPE, "scene_tiles: tile %d larger than the resident %dx%d scene", T, rows, W);
  NG_REQUIRE(((uintptr_t)origins & 7) == 0, NG_E_ALIGN, "scene_tiles: origins must be 8-byte aligned");
  const bool vec = T % 4 == 0;
  NG_REQUIRE(!vec || ((uintptr_t)dst & 15) == 0, NG_E_ALIGN, "scene_tiles: dst must be 16-byte aligned");
  NG_REQUIRE(n <= 65535 && C <= 65535, NG_E_SHAPE, "scene_tiles: at most 65535 windows per call");
  const int per_tile = T * (vec ? T / 4 : T);
  const dim3 grid((per_tile + SC_THREADS - 1) / SC_THREADS, C, n);
  cudaStream_t st = (cudaStream_t)stream;
  const int2* org = reinterpret_cast<const int2*>(origins);
  if (dtype == NG_F32) {
    if (vec) scene_tiles_kernel<float, 4><<<grid, SC_THREADS, 0, st>>>((const float*)scene, C, rows, W, row0, org, T, dn_scale, dst);
    else scene_tiles_kernel<float, 1><<<grid, SC_THREADS, 0, st>>>((const float*)scene, C, rows, W, row0, org, T, dn_scale, dst);
  } else {
    if (vec) scene_tiles_kernel<uint16_t, 4><<<grid, SC_THREADS, 0, st>>>((const uint16_t*)scene, C, rows, W, row0, org, T, dn_scale, dst);
    else scene_tiles_kernel<uint16_t, 1><<<grid, SC_THREADS, 0, st>>>((const uint16_t*)scene, C, rows, W, row0, org, T, dn_scale, dst);
  }
  NG_LAUNCH_CHECK("scene_tiles_kernel");
  return NG_OK;
}

extern "C" int ng_scene_tile_valid(const void* scene, int32_t dtype, int32_t C, int32_t rows, int32_t W, int32_t row0,
                                   const int32_t* origins, int32_t n, int32_t T, float nodata, int32_t* counts,
                                   void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(scene && origins && counts && C > 0 && rows > 0 && W > 0 && row0 >= 0 && n > 0 && T > 0, NG_E_ARG,
             "scene_tile_valid: bad arguments");
  NG_REQUIRE(dtype == NG_F32 || dtype == NG_U16, NG_E_ARG, "scene_tile_valid: the scene must be NG_F32 or NG_U16");
  NG_REQUIRE(((uintptr_t)origins & 7) == 0, NG_E_ALIGN, "scene_tile_valid: origins must be 8-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int2* org = reinterpret_cast<const int2*>(origins);
  if (dtype == NG_F32)
    scene_valid_kernel<float><<<n, SV_THREADS, 0, st>>>((const float*)scene, C, rows, W, row0, org, T, nodata, counts);
  else
    scene_valid_kernel<uint16_t><<<n, SV_THREADS, 0, st>>>((const uint16_t*)scene, C, rows, W, row0, org, T, nodata, counts);
  NG_LAUNCH_CHECK("scene_valid_kernel");
  return NG_OK;
}

static int check_blend(const float* pred, const int32_t* oy, int32_t ny, const int32_t* ox, int32_t nx, int32_t T,
                       int32_t overlap, int32_t W, int32_t y0, int32_t y1, float* out) {
  NG_REQUIRE(pred && oy && ox && out && ny > 0 && nx > 0 && T > 0 && W >= T && y0 >= 0 && y1 > y0, NG_E_ARG,
             "scene_blend: bad arguments");
  NG_REQUIRE(overlap >= 0 && overlap < T, NG_E_ARG, "scene_blend: overlap %d outside [0, %d)", overlap, T);
  return NG_OK;
}

extern "C" int ng_scene_blend(const float* pred, const int32_t* oy, int32_t ny, const int32_t* ox, int32_t nx, int32_t T,
                              int32_t overlap, int32_t W, int32_t y0, int32_t y1, float* out, void* stream) {
  int r = require_sm100(); if (r) return r;
  r = check_blend(pred, oy, ny, ox, nx, T, overlap, W, y0, y1, out); if (r) return r;
  return launch_blend<false, false, false, float>(pred, nullptr, oy, ny, ox, nx, T, overlap, W, y0, y1, SceneMask<float>{},
                                                 SceneIndices{}, out, stream);
}

extern "C" int ng_scene_blend_masked(const float* pred, const int32_t* slot, const int32_t* oy, int32_t ny,
                                     const int32_t* ox, int32_t nx, int32_t T, int32_t overlap, int32_t W, int32_t y0,
                                     int32_t y1, const void* scene, int32_t dtype, int32_t C, int32_t rows,
                                     int32_t row0, float nodata, float nodata_out, float* out, void* stream) {
  int r = require_sm100(); if (r) return r;
  r = check_blend(pred, oy, ny, ox, nx, T, overlap, W, y0, y1, out); if (r) return r;
  NG_REQUIRE(slot && scene && C > 0 && rows > 0 && row0 >= 0, NG_E_ARG, "scene_blend_masked: bad arguments");
  NG_REQUIRE(dtype == NG_F32 || dtype == NG_U16, NG_E_ARG, "scene_blend_masked: the scene must be NG_F32 or NG_U16");
  NG_REQUIRE(row0 <= y0 && y1 <= row0 + rows, NG_E_SHAPE,
             "scene_blend_masked: rows [%d, %d) are not inside the resident scene rows [%d, %d)", y0, y1, row0,
             row0 + rows);
  if (dtype == NG_F32)
    return launch_blend<true, true, false, float>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1,
                                                  SceneMask<float>{(const float*)scene, C, rows, row0, nodata, nodata_out},
                                                  SceneIndices{}, out, stream);
  return launch_blend<true, true, false, uint16_t>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1,
                                                   SceneMask<uint16_t>{(const uint16_t*)scene, C, rows, row0, nodata,
                                                                       nodata_out},
                                                   SceneIndices{}, out, stream);
}

extern "C" int ng_scene_blend_indices(const float* pred, const int32_t* slot, const int32_t* oy, int32_t ny,
                                      const int32_t* ox, int32_t nx, int32_t T, int32_t overlap, int32_t W, int32_t y0,
                                      int32_t y1, const void* scene, int32_t dtype, int32_t C, int32_t rows,
                                      int32_t row0, float dn_scale, int32_t use_nodata, float nodata, float nodata_out,
                                      const int32_t* which, int32_t k, float* out, void* stream) {
  int r = require_sm100(); if (r) return r;
  r = check_blend(pred, oy, ny, ox, nx, T, overlap, W, y0, y1, out); if (r) return r;
  NG_REQUIRE(scene && which && rows > 0 && row0 >= 0, NG_E_ARG, "scene_blend_indices: bad arguments");
  NG_REQUIRE(k >= 1 && k <= SCENE_MAX_INDICES, NG_E_ARG, "scene_blend_indices: k = %d outside [1, %d]", k,
             SCENE_MAX_INDICES);
  SceneIndices idx{};
  for (int i = 0; i < k; ++i) {
    NG_REQUIRE(which[i] >= 1 && which[i] <= 6, NG_E_ARG, "scene_blend_indices: which[%d] = %d outside [1, 6]", i,
               which[i]);
    idx.which[i] = which[i];
  }
  idx.k = k;
  idx.dn_scale = dn_scale;
  NG_REQUIRE(C >= 3, NG_E_ARG, "scene_blend_indices: the scene has %d channels, the indices need R, G, B", C);
  NG_REQUIRE(dtype == NG_F32 || dtype == NG_U16, NG_E_ARG, "scene_blend_indices: the scene must be NG_F32 or NG_U16");
  NG_REQUIRE(dtype != NG_U16 || dn_scale > 0.f, NG_E_ARG, "scene_blend_indices: dn_scale must be positive");
  NG_REQUIRE(row0 <= y0 && y1 <= row0 + rows, NG_E_SHAPE,
             "scene_blend_indices: rows [%d, %d) are not inside the resident scene rows [%d, %d)", y0, y1, row0,
             row0 + rows);
  NG_REQUIRE(((uintptr_t)out & (W % 4 == 0 ? 15 : 3)) == 0, NG_E_ALIGN,
             "scene_blend_indices: out must be %d-byte aligned", W % 4 == 0 ? 16 : 4);
  if (dtype == NG_F32)
    return launch_blend_indices<float>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1,
                                       SceneMask<float>{(const float*)scene, C, rows, row0, nodata, nodata_out},
                                       use_nodata != 0, idx, out, stream);
  return launch_blend_indices<uint16_t>(pred, slot, oy, ny, ox, nx, T, overlap, W, y0, y1,
                                        SceneMask<uint16_t>{(const uint16_t*)scene, C, rows, row0, nodata, nodata_out},
                                        use_nodata != 0, idx, out, stream);
}
