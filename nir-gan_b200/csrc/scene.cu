// Whole-scene inference around the generator: cut overlapping windows of a scene into the generator's NCHW fp32 batch
// layout, and blend the per-tile predictions back into one NIR band.  The reference only runs pre-cut tiles
// (create_synthetic_dataset.py:93,100-118); these two kernels replace the per-tile `model(hr)` loop's hand-written
// cutting and stitching.  Both are HBM-bound single passes; neither uses atomics, so results are bit-reproducible.
//
// Blend (nirgan_b200/scene.py states the same definitions):
//   out(y, x) = sum_t w_t(y, x) p_t(y, x) / sum_t w_t(y, x)   over the tiles t covering (y, x), ascending (k_y, k_x)
//   w(i, j)   = w1(i) w1(j),   w1(i) = min(i + 1, T - i, overlap + 1) / (overlap + 1)
// computed with the integer weights (overlap + 1)^2 w(i, j), and a pixel covered by a single tile takes that tile's value unchanged.
#include "common.cuh"

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

// (overlap + 1) * w1(i): the common factor cancels in the normalised sum, and the integer weights and their sums are
// exact in fp32 (at most (overlap + 1)^2 per tile)
__device__ __forceinline__ int blend_m1(int i, int T, int ov1) { return min(min(i + 1, T - i), ov1); }

// first index k of the ascending origins o[0..n) with o[k] + T > p (the first tile that can cover p)
__device__ __forceinline__ int first_cover(const int* __restrict__ o, int n, int T, int p) {
  int lo = 0, hi = n;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (o[mid] + T <= p) lo = mid + 1; else hi = mid; }
  return lo;
}

// out(y, x) over the covering tiles: rows ky0.. of oy, columns found here (ascending (ky, kx), fp32)
__device__ __forceinline__ float blend_pixel(const float* __restrict__ pred, const int* __restrict__ oy, int ny, int ky0,
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
      last = __ldg(prow + (size_t)kx * T * T + j);
      acc = __fmaf_rn(w, last, acc);
      wsum = __fadd_rn(wsum, w);
      ++cnt;
    }
  }
  return cnt == 1 ? last : __fdiv_rn(acc, wsum);      // no covering tile: 0 / 0 = NaN marks the caller's error
}

// gather form: every output pixel of rows [y0, y0 + rows) reads its covering tiles and is written once.  V consecutive
// pixels of one row per thread (V = 4 when W % 4 == 0: one 16-byte store).
template <int V>
__global__ void __launch_bounds__(SC_THREADS)
scene_blend_kernel(const float* __restrict__ pred, const int* __restrict__ oy, int ny, const int* __restrict__ ox, int nx,
                   int T, int overlap, int W, int y0, int rows, float* __restrict__ out) {
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) * V;
  if (x >= W) return;
  const int ov1 = overlap + 1;
  for (int row = blockIdx.y; row < rows; row += gridDim.y) {
    const int y = y0 + row;
    const int ky0 = first_cover(oy, ny, T, y);
    float* o = out + (size_t)row * W + x;
    if constexpr (V == 4)
      *reinterpret_cast<float4*>(o) = make_float4(blend_pixel(pred, oy, ny, ky0, ox, nx, T, ov1, y, x),
                                                  blend_pixel(pred, oy, ny, ky0, ox, nx, T, ov1, y, x + 1),
                                                  blend_pixel(pred, oy, ny, ky0, ox, nx, T, ov1, y, x + 2),
                                                  blend_pixel(pred, oy, ny, ky0, ox, nx, T, ov1, y, x + 3));
    else
      *o = blend_pixel(pred, oy, ny, ky0, ox, nx, T, ov1, y, x);
  }
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

extern "C" int ng_scene_blend(const float* pred, const int32_t* oy, int32_t ny, const int32_t* ox, int32_t nx, int32_t T,
                              int32_t overlap, int32_t W, int32_t y0, int32_t y1, float* out, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(pred && oy && ox && out && ny > 0 && nx > 0 && T > 0 && W >= T && y0 >= 0 && y1 > y0, NG_E_ARG,
             "scene_blend: bad arguments");
  NG_REQUIRE(overlap >= 0 && overlap < T, NG_E_ARG, "scene_blend: overlap %d outside [0, %d)", overlap, T);
  const bool vec = W % 4 == 0 && ((uintptr_t)out & 15) == 0;
  const int V = vec ? 4 : 1;
  const int per_row = (W + V - 1) / V;
  const dim3 grid((per_row + SC_THREADS - 1) / SC_THREADS, y1 - y0 < 65535 ? y1 - y0 : 65535);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec) scene_blend_kernel<4><<<grid, SC_THREADS, 0, st>>>(pred, oy, ny, ox, nx, T, overlap, W, y0, y1 - y0, out);
  else scene_blend_kernel<1><<<grid, SC_THREADS, 0, st>>>(pred, oy, ny, ox, nx, T, overlap, W, y0, y1 - y0, out);
  NG_LAUNCH_CHECK("scene_blend_kernel");
  return NG_OK;
}
