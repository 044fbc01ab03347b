// Memory-bound kernels of the hot path: layout / packing, InstanceNorm statistics, the fused
// normalise + inject + activation + residual + halo "apply", the SatCLIP projection, the fused
// pixel losses and Adam.  All are vectorised (16-byte accesses on the 16-bit paths) and sized in
// multiples of the SM count.
#include "common.cuh"
#include "rs_index.cuh"
#include <stdlib.h>
#include <type_traits>

namespace ng {

// ---------------------------------------------------------------------------------------------
// weight packing: src fp32 [d0][d1][KH][KW] -> dst [tap][n_pad][k_pad], n = d(n_axis), k = the other
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void pack_weight_kernel(const float* __restrict__ src, int d0, int d1, int taps, int n_axis, int n_pad,
                                   int k_pad, T* __restrict__ dst) {
  const long long total = (long long)taps * n_pad * k_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % k_pad);
    const int n = (int)((i / k_pad) % n_pad);
    const int tp = (int)(i / ((long long)k_pad * n_pad));
    const int a0 = n_axis == 0 ? n : k, a1 = n_axis == 0 ? k : n;
    float v = 0.f;
    if (a0 < d0 && a1 < d1) v = src[((long long)a0 * d1 + a1) * taps + tp];
    dst[i] = from_f32<T>(v);
  }
}

// ConvTranspose2d(k3, s2, p1) weights [Cin][Cout][3][3] -> merged-phase layout [shift][phase*Cout + co][Cin]
template <typename T>
__global__ void pack_phasemerged_kernel(const float* __restrict__ src, int Cin, int Cout, T* __restrict__ dst) {
  const long long total = 4ll * 4 * Cout * Cin;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin);
    long long r = i / Cin;
    const int co = (int)(r % Cout); r /= Cout;
    const int ph = (int)(r % 4), sh = (int)(r / 4);
    // slot ph of the virtual channels = output parity in Gray order (0,0), (0,1), (1,1), (1,0): see conv_tc.cu
    const int pa = ph >> 1, pb = (ph & 1) ^ (ph >> 1), sy = sh >> 1, sx = sh & 1;
    const int kh = pa + 1 - 2 * sy, kw = pb + 1 - 2 * sx;
    float v = 0.f;
    if (kh >= 0 && kh < 3 && kw >= 0 && kw < 3) v = src[(((long long)ci * Cout + co) * 3 + kh) * 3 + kw];
    dst[i] = from_f32<T>(v);
  }
}

__global__ void unpack_wgrad_kernel(const float* __restrict__ packed, int d0, int d1, int taps, int n_axis,
                                    int n_pad, int k_pad, float scale, const float* __restrict__ dev_scale, float beta,
                                    float* __restrict__ dst) {
  const long long total = (long long)d0 * d1 * taps;
  if (dev_scale) scale *= dev_scale[0];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int tp = (int)(i % taps);
    const int a1 = (int)((i / taps) % d1);
    const int a0 = (int)(i / ((long long)taps * d1));
    const int n = n_axis == 0 ? a0 : a1, k = n_axis == 0 ? a1 : a0;
    const float v = scale * packed[((long long)tp * n_pad + n) * k_pad + k];
    dst[i] = beta != 0.f ? fmaf(beta, dst[i], v) : v;
  }
}

// ---------------------------------------------------------------------------------------------
// input preparation: NCHW fp32 (1 or 2 sources) -> haloed NHWC with channel padding
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void prep_input_kernel(const float* __restrict__ sa, int ca, const float* __restrict__ sb, int cb, int B,
                                  int H, int W, int wrap, int halo, int halo_mode, int cpad, T* __restrict__ dst) {
  const int H1 = H + 2 * wrap, W1 = W + 2 * wrap;     // after the wrapper's reflect padding
  const int Hb = H1 + 2 * halo, Wb = W1 + 2 * halo;
  const long long total = (long long)B * Hb * Wb;
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    const int xb = (int)(p % Wb);
    const int yb = (int)((p / Wb) % Hb);
    const int n = (int)(p / ((long long)Wb * Hb));
    int y1 = yb - halo, x1 = xb - halo;
    bool zero = false;
    if (halo_mode == NG_HALO_REFLECT) { y1 = reflect_idx(y1, H1); x1 = reflect_idx(x1, W1); }
    else zero = y1 < 0 || y1 >= H1 || x1 < 0 || x1 >= W1;
    T* o = dst + p * cpad;
    if constexpr (sizeof(T) == 2) if ((cpad & 7) == 0) {   // 16-bit paths: one 16-byte store per 8 channels
      const int y0 = zero ? 0 : reflect_idx(y1 - wrap, H), x0 = zero ? 0 : reflect_idx(x1 - wrap, W);
      for (int c0 = 0; c0 < cpad; c0 += 8) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = c0 + k;
          v[k] = 0.f;
          if (!zero) {
            if (c < ca) v[k] = sa[(((long long)n * ca + c) * H + y0) * W + x0];
            else if (c < ca + cb) v[k] = sb[(((long long)n * cb + (c - ca)) * H + y0) * W + x0];
          }
        }
        uint4 u;
        u.x = pack2<T>(v[0], v[1]); u.y = pack2<T>(v[2], v[3]); u.z = pack2<T>(v[4], v[5]); u.w = pack2<T>(v[6], v[7]);
        *reinterpret_cast<uint4*>(o + c0) = u;
      }
      continue;
    }
    if (zero) {
      for (int c = 0; c < cpad; ++c) o[c] = from_f32<T>(0.f);
      continue;
    }
    const int y0 = reflect_idx(y1 - wrap, H), x0 = reflect_idx(x1 - wrap, W);
    for (int c = 0; c < cpad; ++c) {
      float v = 0.f;
      if (c < ca) v = sa[(((long long)n * ca + c) * H + y0) * W + x0];
      else if (c < ca + cb) v = sb[(((long long)n * cb + (c - ca)) * H + y0) * W + x0];
      o[c] = from_f32<T>(v);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// space-to-depth form of the PatchGAN input layer (Conv2d(4 -> 64, k4, s2, p1), model/networks.py:559):
// the zero-padded (pad 1) image is stored as [B][(H+2)/2][(W+2)/2][(py*2+px)*cs + c] (cs = 16 channel slots per parity),
// on which the 4x4 stride-2 convolution is a 2x2 STRIDE-1 convolution over 64 channels with kernel position
// (kh, kw) = (2*dy + py, 2*dx + px): a bijection, no padded taps.  The thin 16-channel strided form moved 32-byte TMA
// elements through a 16-stage-per-tile pipeline (0.37 ms per 64 images of 256x256 for a 45 us HBM floor); this one is an
// ordinary 64-channel convolution for forward, weight gradient and data gradient alike.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
prep_input_s2d_kernel(const float* __restrict__ sa, int ca, const float* __restrict__ sb, int cb, int B, int H, int W,
                      T* __restrict__ dst) {
  // one thread = one (output pixel, parity) = 16 channel slots = 32 bytes (two 16-byte stores)
  const int Hs = (H + 2) >> 1, Ws = (W + 2) >> 1;
  const long long total = (long long)B * Hs * Ws * 4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int par = (int)(i & 3);
    long long r = i >> 2;
    const int xs = (int)(r % Ws); r /= Ws;
    const int ys = (int)(r % Hs);
    const int n = (int)(r / Hs);
    const int y0 = 2 * ys + (par >> 1) - 1, x0 = 2 * xs + (par & 1) - 1;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    if (y0 >= 0 && y0 < H && x0 >= 0 && x0 < W) {
      for (int c = 0; c < ca; ++c) v[c] = sa[(((long long)n * ca + c) * H + y0) * W + x0];
      for (int c = 0; c < cb; ++c) v[ca + c] = sb[(((long long)n * cb + c) * H + y0) * W + x0];
    }
    uint4 u0, u1;
    u0.x = pack2<T>(v[0], v[1]); u0.y = pack2<T>(v[2], v[3]); u0.z = pack2<T>(v[4], v[5]); u0.w = pack2<T>(v[6], v[7]);
    u1.x = pack2<T>(v[8], v[9]); u1.y = pack2<T>(v[10], v[11]); u1.z = pack2<T>(v[12], v[13]); u1.w = pack2<T>(v[14], v[15]);
    uint4* o = reinterpret_cast<uint4*>(dst + i * 16);
    o[0] = u0; o[1] = u1;
  }
}

// weights of the space-to-depth form.  src fp32 [O][I][4][4]; tap = dy*2 + dx, element (py*2+px)*16 + c <-> w[o][c][2dy+py][2dx+px].
// transpose == 0: dst [tap][O][64] (forward);  transpose == 1: dst [tap][64][O] (data gradient: n = input slot, k = O)
template <typename T>
__global__ void pack_weight_s2d_kernel(const float* __restrict__ src, int O, int I, int transpose, T* __restrict__ dst) {
  const int total = 4 * O * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int e, o, tap;
    if (!transpose) { e = i & 63; o = (i >> 6) % O; tap = (i >> 6) / O; }
    else { o = i % O; e = (i / O) & 63; tap = (i / O) >> 6; }
    const int par = e >> 4, c = e & 15;
    const int kh = 2 * (tap >> 1) + (par >> 1), kw = 2 * (tap & 1) + (par & 1);
    float v = 0.f;
    if (c < I) v = src[(((long long)o * I + c) * 4 + kh) * 4 + kw];
    dst[i] = from_f32<T>(v);
  }
}

// inverse for gradients: packed fp32 [tap][O][64] -> dst fp32 [O][I][4][4] (dst = beta * dst + scale * dev_scale[0] * packed)
__global__ void unpack_wgrad_s2d_kernel(const float* __restrict__ packed, int O, int I, float scale,
                                        const float* __restrict__ dev_scale, float beta, float* __restrict__ dst) {
  const int total = O * I * 16;
  if (dev_scale) scale *= dev_scale[0];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int kw = i & 3, kh = (i >> 2) & 3, c = (i >> 4) % I, o = (i >> 4) / I;
    const int tap = (kh >> 1) * 2 + (kw >> 1), par = (kh & 1) * 2 + (kw & 1);
    const float v = scale * packed[((long long)tap * O + o) * 64 + par * 16 + c];
    dst[i] = beta != 0.f ? fmaf(beta, dst[i], v) : v;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
in_stats_kernel(const T* __restrict__ y, int HW, int C, float* __restrict__ mr) {
  __shared__ float red[8][33];
  __shared__ float smean[32];
  const int n = blockIdx.x, c = blockIdx.y * 32 + (threadIdx.x & 31), rg = threadIdx.x >> 5;
  const T* base = y + (size_t)n * HW * C;
  float s = 0.f;
  if (c < C) for (int p = rg; p < HW; p += 8) s += to_f32<T>(base[(size_t)p * C + c]);
  red[rg][threadIdx.x & 31] = s;
  __syncthreads();
  if (rg == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; ++i) tsum += red[i][threadIdx.x];
    smean[threadIdx.x] = tsum / HW;
  }
  __syncthreads();
  const float mean = smean[threadIdx.x & 31];
  float q = 0.f;
  if (c < C) for (int p = rg; p < HW; p += 8) { float d = to_f32<T>(base[(size_t)p * C + c]) - mean; q += d * d; }
  red[rg][threadIdx.x & 31] = q;
  __syncthreads();
  if (rg == 0 && c < C) {
    float tq = 0.f;
    for (int i = 0; i < 8; ++i) tq += red[i][threadIdx.x];
    mr[((size_t)n * C + c) * 2 + 0] = mean;
    mr[((size_t)n * C + c) * 2 + 1] = rsqrtf(tq / HW + 1e-5f);
  }
}

// partials: [B][slots][C][2] (sum, sumsq) -> mean / rstd.  One warp per (n, channel pair): lanes stride over the
// slots, then a fixed-order shuffle tree -> deterministic, and the loads of a warp are independent.
__global__ void __launch_bounds__(256)
in_stats_finalize_kernel(const float* __restrict__ part, int B, int slots, int C, float inv_count,
                         float* __restrict__ mr) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int C2 = C >> 1;
  if (wid >= B * C2) return;
  const int n = wid / C2, c2 = wid % C2;
  const float4* p = reinterpret_cast<const float4*>(part + ((size_t)n * slots * C + 2 * c2) * 2);
  const size_t stride = (size_t)C * 2 / 4;
  float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
  for (int k = lane; k < slots; k += 32) {
    const float4 v = p[(size_t)k * stride];
    s0 += v.x; q0 += v.y; s1 += v.z; q1 += v.w;
  }
  s0 = warp_sum(s0); q0 = warp_sum(q0); s1 = warp_sum(s1); q1 = warp_sum(q1);
  if (lane == 0) {
    const float m0 = s0 * inv_count, m1 = s1 * inv_count;
    const float v0 = fmaxf(q0 * inv_count - m0 * m0, 0.f), v1 = fmaxf(q1 * inv_count - m1 * m1, 0.f);
    *reinterpret_cast<float4*>(mr + ((size_t)n * C + 2 * c2) * 2) =
        make_float4(m0, rsqrtf(v0 + 1e-5f), m1, rsqrtf(v1 + 1e-5f));
  }
}

// ---------------------------------------------------------------------------------------------
// apply: out(haloed) = act( inject( (y-mean)*rstd ) ) + residual
// one thread = one output buffer position x 8 channels (16 B on the 16-bit paths)
// ---------------------------------------------------------------------------------------------
template <typename T> struct Vec8 { T v[8]; };

template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&f)[8]) {
  if constexpr (sizeof(T) == 2) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    float2 a = unpack2<T>(u.x), b = unpack2<T>(u.y), c = unpack2<T>(u.z), d = unpack2<T>(u.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
  } else {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
}
template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&f)[8]) {
  if constexpr (sizeof(T) == 2) {
    uint4 u;
    u.x = pack2<T>(f[0], f[1]); u.y = pack2<T>(f[2], f[3]); u.z = pack2<T>(f[4], f[5]); u.w = pack2<T>(f[6], f[7]);
    *reinterpret_cast<uint4*>(p) = u;
  } else {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
  }
}

__device__ __forceinline__ float bilerp128(const float* __restrict__ e, int oy, int ox, int H, int W) {
  // F.interpolate(mode='bilinear', align_corners=False) from a 128x128 grid (model/generator_inject.py:116)
  const float sy = fmaxf((oy + 0.5f) * (128.f / H) - 0.5f, 0.f), sx = fmaxf((ox + 0.5f) * (128.f / W) - 0.5f, 0.f);
  const int y0 = min((int)sy, 127), x0 = min((int)sx, 127);
  const int y1 = min(y0 + 1, 127), x1 = min(x0 + 1, 127);
  const float ly = sy - y0, lx = sx - x0;
  const float v00 = e[y0 * 128 + x0], v01 = e[y0 * 128 + x1], v10 = e[y1 * 128 + x0], v11 = e[y1 * 128 + x1];
  return (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
}

// Streaming loads / stores: every activation byte is touched exactly once by this kernel, so keep it out of L1.
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

template <typename T>
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a = unpack2<T>(u.x), b = unpack2<T>(u.y), c = unpack2<T>(u.z), d = unpack2<T>(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

// Flat apply.  Block (chunk, n) owns `ppb` consecutive pixels of image n's haloed output buffer (row-major over
// (H+2p) x (W+2p), so its stores are one contiguous span); thread t keeps the channel group c8 = t mod C/8 for its whole
// life (C/8 is a power of two <= 256), so the 8 (mean, rstd) pairs live in registers.  The inner loop is: UNROLL
// independent 16-byte streaming loads (+ residual loads) -> math one pixel at a time -> 16-byte stores.  The pixel ->
// (row, column) split uses a multiply-shift by the precomputed reciprocal of the buffer width.
// DRAM -> L2 bulk prefetch of the source rows a block is about to read (y and, if present, the haloed residual): the
// block's 16-byte loads then see L2 latency, and the bytes a block keeps in flight stop bounding the kernel.  One thread
// per block; rows are over-approximated at the reflect borders (a neighbouring block needs them anyway).
__device__ __forceinline__ void apply_prefetch_rows(const void* y, const void* res, int n, int H, int W, int C, int esz,
                                                    int op, bool reflect, int res_pad, int Wo, int p_begin, int p_end) {
  const int yo0 = p_begin / Wo, yo1 = (p_end - 1) / Wo;
  int lo = min(max(yo0 - op, 0), H - 1), hi = min(max(yo1 - op, 0), H - 1);
  if (reflect) {
    if (yo0 < op) hi = max(hi, min(op, H - 1));
    if (yo1 >= H + op) lo = min(lo, max(H - 1 - op, 0));
  }
  const size_t row = (size_t)W * C * esz;
  const char* yp = reinterpret_cast<const char*>(y) + ((size_t)n * H + lo) * row;
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(yp), "r"((uint32_t)((hi - lo + 1) * row)) : "memory");
  if (res) {
    const size_t rrow = (size_t)(W + 2 * res_pad) * C * esz;
    const char* rp = reinterpret_cast<const char*>(res) + ((size_t)n * (H + 2 * res_pad) + lo + res_pad) * rrow;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(rp), "r"((uint32_t)((hi - lo + 1) * rrow)) : "memory");
  }
}

template <typename T, int UNROLL, bool HAS_RES, bool HAS_INJ>
__global__ void __launch_bounds__(256, 3)
in_apply_kernel(const T* __restrict__ y, int H, int W, int C, int c8_shift, const float* __restrict__ mr,
                const long long* __restrict__ acc, float* __restrict__ mr_out, int act,
                float slope, const T* __restrict__ res, int res_pad, const float* __restrict__ inj, int inj_mode,
                const float* __restrict__ inj_scale, T* __restrict__ out, int op, int halo_mode, int ppb,
                unsigned long long wo_magic, int pf) {
  const int Ho = H + 2 * op, Wo = W + 2 * op, C8 = C >> 3;
  const int n = blockIdx.y;
  const int npix = Ho * Wo;
  const float s = (HAS_INJ && inj_scale) ? *inj_scale : 1.f;
  const int c8 = threadIdx.x & (C8 - 1);
  const int pstep = 256 >> c8_shift;                 // pixels covered by the block per load
  const int p_begin = blockIdx.x * ppb, p_end = min(npix, p_begin + ppb);
  if (pf && threadIdx.x == 0 && p_begin < p_end)
    apply_prefetch_rows(y, HAS_RES ? res : nullptr, n, H, W, C, (int)sizeof(T), op, halo_mode == NG_HALO_REFLECT, res_pad, Wo,
                        p_begin, p_end);
  float mean[8], rstd[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { mean[k] = 0.f; rstd[k] = 1.f; }
  if (mr) {
    const float4* m4 = reinterpret_cast<const float4*>(mr + ((size_t)n * C + c8 * 8) * 2);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 m = m4[k];
      mean[2 * k] = m.x; rstd[2 * k] = m.y; mean[2 * k + 1] = m.z; rstd[2 * k + 1] = m.w;
    }
  } else if (acc) {
    // fixed-point (sum, sum of squares) accumulated by the conv epilogue's integer atomics: exact totals -> mean / rstd
    const longlong2* a2 = reinterpret_cast<const longlong2*>(acc + ((size_t)n * C + c8 * 8) * 2);
    const double inv_n = 1.0 / ((double)H * (double)W);
    const double ks = inv_n / (double)(1 << NG_STAT_SUM_SHIFT), kq = inv_n / (double)(1 << NG_STAT_SQ_SHIFT);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const longlong2 v = a2[k];
      const double m = (double)v.x * ks;
      const double var = fmax((double)v.y * kq - m * m, 0.0);
      mean[k] = (float)m;
      rstd[k] = rsqrtf((float)var + 1e-5f);
    }
    if (mr_out != nullptr && blockIdx.x == 0 && (threadIdx.x >> c8_shift) == 0) {
      float4* o4 = reinterpret_cast<float4*>(mr_out + ((size_t)n * C + c8 * 8) * 2);
#pragma unroll
      for (int k = 0; k < 4; ++k) o4[k] = make_float4(mean[2 * k], rstd[2 * k], mean[2 * k + 1], rstd[2 * k + 1]);
    }
  }
  const bool norm = mr != nullptr || acc != nullptr;
  const int Wr = W + 2 * res_pad;
  const T* ybase = y + (size_t)n * H * W * C + c8 * 8;
  const T* rbase = HAS_RES ? res + ((size_t)n * (H + 2 * res_pad) * Wr + (size_t)res_pad * Wr + res_pad) * C + c8 * 8 : nullptr;
  T* obase = out + (size_t)n * npix * C + c8 * 8;
  const float* injn = HAS_INJ ? inj + (size_t)n * 128 * 128 : nullptr;
  for (int p0 = p_begin + (threadIdx.x >> c8_shift); p0 < p_end; p0 += pstep * UNROLL) {
    // phase 1: issue every load of this batch before any use
    uint4 raw[UNROLL], rres[HAS_RES ? UNROLL : 1];
    float4 rawf[sizeof(T) == 4 ? UNROLL : 1][2], rresf[(sizeof(T) == 4 && HAS_RES) ? UNROLL : 1][2];
    int ysrc[UNROLL], xsrc[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int pp = p0 + u * pstep;
      const int yo = (int)(((unsigned long long)(unsigned)pp * wo_magic) >> 40);
      const int xo = pp - yo * Wo;
      int ys = yo - op, xs = xo - op;
      bool ok = pp < p_end;
      if (halo_mode == NG_HALO_REFLECT) { ys = reflect_idx(ys, H); xs = reflect_idx(xs, W); }
      else ok = ok && ys >= 0 && ys < H && xs >= 0 && xs < W;
      ysrc[u] = ys; xsrc[u] = ok ? xs : -1;
      if (ok) {
        const size_t off = ((size_t)ys * W + xs) * C;
        if constexpr (sizeof(T) == 2) {
          raw[u] = ldg_stream16(ybase + off);
          if constexpr (HAS_RES) rres[u] = ldg_stream16(rbase + ((size_t)ys * Wr + xs) * C);
        } else {
          rawf[u][0] = *reinterpret_cast<const float4*>(ybase + off);
          rawf[u][1] = *reinterpret_cast<const float4*>(ybase + off + 4);
          if constexpr (HAS_RES) {
            rresf[u][0] = *reinterpret_cast<const float4*>(rbase + ((size_t)ys * Wr + xs) * C);
            rresf[u][1] = *reinterpret_cast<const float4*>(rbase + ((size_t)ys * Wr + xs) * C + 4);
          }
        }
      }
    }
    // phase 2: one pixel at a time (small live register set: occupancy is what hides HBM latency)
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int pp = p0 + u * pstep;
      if (pp >= p_end) continue;
      float f[8];
      if (xsrc[u] < 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = 0.f;
      } else {
        if constexpr (sizeof(T) == 2) unpack8<T>(raw[u], f);
        else {
          f[0] = rawf[u][0].x; f[1] = rawf[u][0].y; f[2] = rawf[u][0].z; f[3] = rawf[u][0].w;
          f[4] = rawf[u][1].x; f[5] = rawf[u][1].y; f[6] = rawf[u][1].z; f[7] = rawf[u][1].w;
        }
        if (norm) {
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] = (f[k] - mean[k]) * rstd[k];
        }
        if constexpr (HAS_INJ) {
          const float ev = bilerp128(injn, ysrc[u], xsrc[u], H, W);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            if (inj_mode == NG_INJECT_ADD) f[k] = f[k] + s * ev;
            else if (inj_mode == NG_INJECT_MUL_SCALED) f[k] = f[k] * (1.f + s * ev);
            else f[k] = f[k] * ev;
          }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = apply_act(f[k], act, slope);
        if constexpr (HAS_RES) {
          float rv[8];
          if constexpr (sizeof(T) == 2) unpack8<T>(rres[u], rv);
          else {
            rv[0] = rresf[u][0].x; rv[1] = rresf[u][0].y; rv[2] = rresf[u][0].z; rv[3] = rresf[u][0].w;
            rv[4] = rresf[u][1].x; rv[5] = rresf[u][1].y; rv[6] = rresf[u][1].z; rv[7] = rresf[u][1].w;
          }
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] += rv[k];
        }
      }
      store8<T>(obase + (size_t)pp * C, f);
    }
  }
}

// Lean form of the flat apply for the common case -- 16-bit storage, normalised unit, ReLU or no activation, optional
// residual, no injection -- written for INSTRUCTION count: the generic kernel above executes ~70 warp instructions per
// 16-byte item (ncu r2h: 45 % integer / address arithmetic, IPC 2.0, 51 % of DRAM peak) and is bound by issue slots and
// SM clock (it loses 24 % under the power cap), not by HBM.  Here: (y - mean) * rstd is one FFMA with precomputed
// (rstd, -mean * rstd); ReLU runs on the packed 16-bit result (max with 0 commutes with rounding: same bits); the
// (row, column) of a pixel is advanced incrementally instead of by a 64-bit multiply-shift per pixel; offsets are 32-bit
// element indices added to per-image base pointers.
__device__ __forceinline__ uint32_t relu_packed(uint32_t w, bool bf16) {
  if (bf16) {
    __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&w);
    v = __hmax2(v, __floats2bfloat162_rn(0.f, 0.f));
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __half2 v = *reinterpret_cast<__half2*>(&w);
  v = __hmax2(v, __floats2half2_rn(0.f, 0.f));
  return *reinterpret_cast<uint32_t*>(&v);
}

template <typename T, int UNROLL, bool HAS_RES, bool RELU, int MINB = 3, bool INJ = false>
__global__ void __launch_bounds__(256, MINB)
in_apply_fast_kernel(const T* __restrict__ y, int H, int W, int C, int c8_shift, const float* __restrict__ mr,
                     const long long* __restrict__ acc, float* __restrict__ mr_out, const T* __restrict__ res,
                     int res_pad, T* __restrict__ out, int op, int reflect, int ppb, int pf,
                     const float* __restrict__ inj = nullptr, int inj_mode = 0, const float* __restrict__ inj_scale = nullptr) {
  static_assert(sizeof(T) == 2, "16-bit storage only");
  constexpr bool BF = std::is_same<T, __nv_bfloat16>::value;
  const int Ho = H + 2 * op, Wo = W + 2 * op, C8 = C >> 3;
  const int n = blockIdx.y;
  const int npix = Ho * Wo;
  const int c8 = threadIdx.x & (C8 - 1);
  const int pstep = 256 >> c8_shift;                 // pixels covered by the block per load
  const int p_begin = blockIdx.x * ppb, p_end = min(npix, p_begin + ppb);
  if (pf && threadIdx.x == 0 && p_begin < p_end)
    apply_prefetch_rows(y, HAS_RES ? res : nullptr, n, H, W, C, 2, op, reflect != 0, res_pad, Wo, p_begin, p_end);
  float sa[8], sb[8];                                // xh = y * sa + sb
  if (mr) {
    const float4* m4 = reinterpret_cast<const float4*>(mr + ((size_t)n * C + c8 * 8) * 2);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 m = m4[k];
      sa[2 * k] = m.y; sb[2 * k] = -m.x * m.y; sa[2 * k + 1] = m.w; sb[2 * k + 1] = -m.z * m.w;
    }
  } else {
    const longlong2* a2 = reinterpret_cast<const longlong2*>(acc + ((size_t)n * C + c8 * 8) * 2);
    const double inv_n = 1.0 / ((double)H * (double)W);
    const double ks = inv_n / (double)(1 << NG_STAT_SUM_SHIFT), kq = inv_n / (double)(1 << NG_STAT_SQ_SHIFT);
    float mean[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const longlong2 v = a2[k];
      const double m = (double)v.x * ks;
      const double var = fmax((double)v.y * kq - m * m, 0.0);
      mean[k] = (float)m;
      sa[k] = rsqrtf((float)var + 1e-5f);
      sb[k] = -mean[k] * sa[k];
    }
    if (mr_out != nullptr && blockIdx.x == 0 && (threadIdx.x >> c8_shift) == 0) {
      float4* o4 = reinterpret_cast<float4*>(mr_out + ((size_t)n * C + c8 * 8) * 2);
#pragma unroll
      for (int k = 0; k < 4; ++k) o4[k] = make_float4(mean[2 * k], sa[2 * k], mean[2 * k + 1], sa[2 * k + 1]);
    }
  }
  const int Wr = W + 2 * res_pad;
  const T* ybase = y + (size_t)n * H * W * C + c8 * 8;
  const T* rbase = HAS_RES ? res + ((size_t)n * (H + 2 * res_pad) * Wr + (size_t)res_pad * Wr + res_pad) * C + c8 * 8 : nullptr;
  T* obase = out + (size_t)n * npix * C + c8 * 8;
  // this thread's first pixel -> (row, column) once; afterwards advanced by pstep per unrolled item
  int pp = p_begin + (threadIdx.x >> c8_shift);
  int yo = pp / Wo, xo = pp - yo * Wo;
  const int adv_y = pstep / Wo, adv_x = pstep - adv_y * Wo;      // pstep pixels = adv_y rows + adv_x columns
  // SatCLIP injection (the d1 unit): u = xh * (1 + s * e) | xh + s * e | xh * e with e the bilinear sample of the
  // 128 x 128 embedding map at the SOURCE pixel (generator_inject.py:113-127)
  const float* injn = INJ ? inj + (size_t)n * 128 * 128 : nullptr;
  const float inj_s = (INJ && inj_scale) ? *inj_scale : 1.f;
  while (pp < p_end) {
    uint4 raw[UNROLL], rres[HAS_RES ? UNROLL : 1];
    int ok[UNROLL];
    int ooff[UNROLL];
    int ysrc[INJ ? UNROLL : 1], xsrc[INJ ? UNROLL : 1];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      int ys = yo - op, xs = xo - op;
      bool inside = pp < p_end;
      if (reflect) {
        ys = ys < 0 ? -ys : (ys >= H ? 2 * (H - 1) - ys : ys);
        xs = xs < 0 ? -xs : (xs >= W ? 2 * (W - 1) - xs : xs);
      } else {
        inside = inside && (unsigned)ys < (unsigned)H && (unsigned)xs < (unsigned)W;
      }
      ok[u] = pp < p_end ? (inside ? 1 : 2) : 0;                 // 1 = compute, 2 = zero halo, 0 = past the block
      ooff[u] = pp * C;
      if constexpr (INJ) { ysrc[u] = ys; xsrc[u] = xs; }
      if (inside) {
        raw[u] = ldg_stream16(ybase + (ys * W + xs) * C);
        if constexpr (HAS_RES) rres[u] = ldg_stream16(rbase + (ys * Wr + xs) * C);
      }
      pp += pstep; yo += adv_y; xo += adv_x;
      if (xo >= Wo) { xo -= Wo; ++yo; }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      if (ok[u] == 0) continue;
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (ok[u] == 1) {
        float f[8];
        unpack8<T>(raw[u], f);
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = fmaf(f[k], sa[k], sb[k]);
        if constexpr (INJ) {
          const float ev = bilerp128(injn, ysrc[u], xsrc[u], H, W);
          const float fac = inj_mode == NG_INJECT_MUL_SCALED ? 1.f + inj_s * ev : (inj_mode == NG_INJECT_MUL ? ev : 1.f);
          const float add = inj_mode == NG_INJECT_ADD ? inj_s * ev : 0.f;
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] = fmaf(f[k], fac, add);
        }
        if constexpr (HAS_RES) {
          float rv[8];
          unpack8<T>(rres[u], rv);
          if constexpr (RELU) {
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] = fmaxf(f[k], 0.f) + rv[k];
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] += rv[k];
          }
        }
        o.x = pack2<T>(f[0], f[1]); o.y = pack2<T>(f[2], f[3]); o.z = pack2<T>(f[4], f[5]); o.w = pack2<T>(f[6], f[7]);
        if constexpr (RELU && !HAS_RES) {
          o.x = relu_packed(o.x, BF); o.y = relu_packed(o.y, BF); o.z = relu_packed(o.z, BF); o.w = relu_packed(o.w, BF);
        }
      }
      *reinterpret_cast<uint4*>(obase + ooff[u]) = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// linear: y[b][n] = x[b][:] . w[n][:] + bias[n]; one warp per n, lanes split K, loop over b
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
linear_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias, int B, int K,
              int N, float* __restrict__ y) {
  // tile: 64 batch rows x 64 outputs, K in chunks of 32; thread = 4 x 4 outputs
  __shared__ float Xs[32][64 + 4];
  __shared__ float Ws[32][64 + 4];
  const int n0 = blockIdx.x * 64, b0 = blockIdx.y * 64;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int lr = t >> 2, lk = (t & 3) * 8;      // loader: 64 rows x 4 threads x 8 k
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + lk + e;
      Xs[lk + e][lr] = (b0 + lr < B && k < K) ? x[(size_t)(b0 + lr) * K + k] : 0.f;
      Ws[lk + e][lr] = (n0 + lr < N && k < K) ? w[(size_t)(n0 + lr) * K + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = Xs[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Ws[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) y[(size_t)b * N + n] = acc[i][j] + (bias ? bias[n] : 0.f);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// losses
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
lsgan_kernel(const float* __restrict__ p, long long n, float target, float* __restrict__ partial,
             float* __restrict__ grad, float gcoef) {
  float s = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float d = p[i] - target;
    s += d * d;
    if (grad) grad[i] = gcoef * d;
  }
  __shared__ float red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; ++i) tsum += red[i];
    partial[blockIdx.x] = tsum;
  }
}

// deterministic second stage: out[j] (+)= scale * sum_i partial[i*stride + j]
__global__ void reduce_partials_kernel(const float* __restrict__ partial, int nblocks, int stride, float scale,
                                       float* __restrict__ out, int accumulate) {
  const int j = threadIdx.x;
  if (j >= stride) return;
  double s = 0.0;
  for (int i = 0; i < nblocks; ++i) s += partial[(size_t)i * stride + j];
  const float v = (float)(s * scale);
  out[j] = accumulate ? out[j] + v : v;
}

// ---------------------------------------------------------------------------------------------
// All of RemoteSensingIndices (utils/remote_sensing_indices.py:84-319) + the pix2pix L1 term in one pass.
// term order: 0 = L1(pred, nir), 1 = NDVI, 2 = NDWI, 3 = GNDVI, 4 = SAVI, 5 = MSAVI, 6 = EVI (the reference's iteration
// order, :45-52).  `mask` selects the terms to evaluate (the kernel is ALU-bound once all six indices are on);
// criterion 0 = l1 (F.l1_loss), 1 = l2 (F.mse_loss) for the six indices.  Also writes
// dpred = d( sum_i w_i * term_i ) / dpred.  The per-pixel formulas (RsPix, rs_ndvi ..) are in rs_index.cuh.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float sgn(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }

struct RsWeights { float w[7]; };

__global__ void __launch_bounds__(256)
rs_pixel_loss_kernel(const float* __restrict__ rgb, const float* __restrict__ nir, const float* __restrict__ pred,
                     int B, int HW, RsWeights wt, const float* __restrict__ wdev, int criterion, int mask, float inv_n,
                     float* __restrict__ partial, float* __restrict__ dpred) {
  if (wdev) {                 // weights known only on the device (autograd's upstream gradient per term)
#pragma unroll
    for (int k = 0; k < 7; ++k) wt.w[k] = wdev[k];
  }
  float acc[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) acc[k] = 0.f;
  const long long total = (long long)B * HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / HW), q = (int)(i % HW);
    const float R = rgb[((size_t)n * 3 + 0) * HW + q], G = rgb[((size_t)n * 3 + 1) * HW + q],
                Bl = rgb[((size_t)n * 3 + 2) * HW + q];
    const float t = nir[i], p = pred[i];
    float g = 0.f;
    if (mask & 1) {
      const float d0 = p - t;
      acc[0] += fabsf(d0);
      g += wt.w[0] * sgn(d0);
    }
    auto term = [&](int k, const RsPix& x) {
      const float df = x.it - x.ip;
      if (criterion == 0) { acc[k] += fabsf(df); g += wt.w[k] * (-sgn(df)) * x.dip; }
      else { acc[k] = fmaf(df, df, acc[k]); g += wt.w[k] * (-2.f * df) * x.dip; }
    };
    if (mask & 2) term(1, rs_ndvi(t, p, R, 1e-6f));
    if (mask & 4) term(2, rs_ndvi(t, p, G, 1e-6f));
    if (mask & 8) term(3, rs_gndvi(t, p, R, G));
    if (mask & 16) term(4, rs_savi(t, p, R));
    if (mask & 32) term(5, rs_msavi(t, p, R));
    if (mask & 64) term(6, rs_evi(t, p, R, Bl, 1e-6f));
    if (dpred) dpred[i] = g * inv_n;
  }
  __shared__ float red[7][8];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const float v = warp_sum(acc[k]);
    if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    float tsum = 0.f;
    if (threadIdx.x < 7)
      for (int i = 0; i < 8; ++i) tsum += red[threadIdx.x][i];
    partial[(size_t)blockIdx.x * 8 + threadIdx.x] = tsum;
  }
}

// 'index' mode of RemoteSensingIndices: the index maps themselves (target, prediction); eps as in the reference
// (loss_eps != 0 reproduces the loss-mode epsilons, 0 the index-mode formulas)
__global__ void __launch_bounds__(256)
rs_index_kernel(const float* __restrict__ rgb, const float* __restrict__ nir, const float* __restrict__ pred, int B,
                int HW, int which, int loss_eps, float* __restrict__ out_t, float* __restrict__ out_p) {
  const long long total = (long long)B * HW;
  const float eps = loss_eps ? 1e-6f : 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / HW), q = (int)(i % HW);
    const float R = rgb[((size_t)n * 3 + 0) * HW + q], G = rgb[((size_t)n * 3 + 1) * HW + q],
                Bl = rgb[((size_t)n * 3 + 2) * HW + q];
    const float t = nir[i], p = pred[i];
    RsPix x;
    switch (which) {
      case 1: x = rs_ndvi(t, p, R, eps); break;
      case 2: x = rs_ndvi(t, p, G, eps); break;
      case 3: x = rs_gndvi(t, p, R, G); break;
      case 4: x = rs_savi(t, p, R); break;
      case 5: x = rs_msavi(t, p, R); break;
      default: x = rs_evi(t, p, R, Bl, eps); break;
    }
    out_t[i] = x.it;
    out_p[i] = x.ip;
  }
}

// ---------------------------------------------------------------------------------------------
// Adam
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
            long long n, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float gscale) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    // torch.optim.Adam (single-tensor): denom = sqrt(v)/sqrt(bc2) + eps; p -= lr/bc1 * m/denom
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}


// Multi-tensor Adam over a flat gradient / moment arena: parameter tensors stay where the nn.Module keeps them (table of
// pointers + element offsets into the arena), so one launch updates every parameter of an optimizer.  `skip` (device
// flag, e.g. "a gradient is not finite") turns the launch into a no-op without a host round trip.
__global__ void __launch_bounds__(256)
adam_multi_kernel(float* const* __restrict__ params, const long long* __restrict__ offsets,
                  const long long* __restrict__ numel, int ntensors, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long total, float lr,
                  float b1, float b2, float eps, float gscale, const int* __restrict__ step_dev,
                  const int* __restrict__ skip) {
  if (skip && *skip) return;
  // bias corrections from the device-side step counter (already advanced for this step by adam_advance_kernel)
  const float stepf = (float)(*step_dev);
  const float bc1 = 1.f - powf(b1, stepf), bc2_sqrt = sqrtf(1.f - powf(b2, stepf));
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int lo = 0, hi = ntensors - 1;                       // last tensor whose offset <= i
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (offsets[mid] <= i) lo = mid; else hi = mid - 1; }
    const long long j = i - offsets[lo];
    if (j >= numel[lo]) continue;                        // alignment padding between arena slots: no parameter behind it
    float* p = params[lo] + j;
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    *p -= (lr / bc1) * (mi / denom);
  }
}

__global__ void adam_advance_kernel(int* __restrict__ step_dev, const int* __restrict__ skip) {
  if (!(skip && *skip)) *step_dev += 1;
}

// flag[0] = 1 if any element of x is inf / NaN (flag must be zeroed by the caller's memset, done in the entry point)
__global__ void __launch_bounds__(256)
nonfinite_flag_kernel(const float* __restrict__ x, long long n, int* __restrict__ flag) {
  bool bad = false;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    bad |= (__float_as_uint(x[i]) & 0x7f800000u) == 0x7f800000u;
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// ---------------------------------------------------------------------------------------------
// generator stem in row-merged form (see ng_prep_stem in the header): one thread = one 16-byte
// (kw, 8-channel) group of one output pixel.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
prep_stem_kernel(const float* __restrict__ src, int cin, int B, int H, int W, int wrap, int halo, int KW,
                 T* __restrict__ dst) {
  // block = one output row (n, yb): no per-item division; item = (x, kw) -> 16 bytes; consecutive threads write
  // consecutive 16-byte groups and read consecutive source columns
  const int H1 = H + 2 * wrap, W1 = W + 2 * wrap, Hb = H1 + 2 * halo;
  const int row = blockIdx.x;
  const int yb = row % Hb, n = row / Hb;
  const int y0 = reflect_idx(reflect_idx(yb - halo, H1) - wrap, H);
  const float* srow = src + ((size_t)n * cin * H + y0) * W;
  const size_t plane = (size_t)H * W;
  T* drow = dst + (size_t)row * W1 * 64;
  for (int i = threadIdx.x; i < W1 * 8; i += 256) {
    const int kw = i & 7, x = i >> 3;
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) f[c] = 0.f;
    if (kw < KW) {
      // column x + kw of the (halo-padded) image = column (x + kw - halo) of the wrapper-padded image
      const int x0 = reflect_idx(reflect_idx(x + kw - halo, W1) - wrap, W);
      for (int c = 0; c < cin; ++c) f[c] = srow[c * plane + x0];
    }
    T* o = drow + (size_t)i * 8;
    if constexpr (sizeof(T) == 2) {
      uint4 u;
      u.x = pack2<T>(f[0], f[1]); u.y = pack2<T>(f[2], f[3]); u.z = pack2<T>(f[4], f[5]); u.w = pack2<T>(f[6], f[7]);
      *reinterpret_cast<uint4*>(o) = u;
    } else {
      *reinterpret_cast<float4*>(o) = make_float4(f[0], f[1], f[2], f[3]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(f[4], f[5], f[6], f[7]);
    }
  }
}

template <typename T>
__global__ void pack_rowmerged_kernel(const float* __restrict__ src, int O, int I, int KH, int KW, int cs,
                                      T* __restrict__ dst) {
  const int RW = 8 * cs;                               // row width: 64 (c_slots 8) or 32 (c_slots 4)
  const int total = KH * O * RW;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i % RW, o = (i / RW) % O, kh = (i / RW) / O;
    const int kw = e / cs, c = e % cs;
    float v = 0.f;
    if (kw < KW && c < I) v = src[(((long long)o * I + c) * KH + kh) * KW + kw];
    dst[i] = from_f32<T>(v);
  }
}

__global__ void unpack_rowmerged_kernel(const float* __restrict__ packed, int O, int I, int KH, int KW, float scale,
                                        const float* __restrict__ dev_scale, float beta, float* __restrict__ dst) {
  const int total = O * I * KH * KW;
  if (dev_scale) scale *= dev_scale[0];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int kw = i % KW, kh = (i / KW) % KH, c = (i / (KW * KH)) % I, o = i / (KW * KH * I);
    const float v = scale * packed[((long long)kh * O + o) * 64 + kw * 8 + c];
    dst[i] = beta != 0.f ? fmaf(beta, dst[i], v) : v;
  }
}

// ---------------------------------------------------------------------------------------------
// tap gather: out[n][y][x] = act(bias + sum_t z[n][y+kh][x+kw][t])   (see ng_tap_gather)
// one warp = 32 consecutive output columns of one row; lanes walk the taps.
// ---------------------------------------------------------------------------------------------
// block = 8 x 32 output pixels; the (8+KH-1) x (32+KW-1) input pixels' tap vectors are staged in shared memory
// (one warp copies one pixel's 128-byte vector per step -> fully coalesced; pixel pitch ZW+1 words -> the strided
// reads below are bank-conflict free), then each thread sums its KH*KW taps.  KH, KW, ZC are compile-time.
constexpr int TG_H = 8, TG_W = 32;
template <typename T, int KH, int KW, int ZC>
__global__ void __launch_bounds__(256)
tap_gather_kernel(const T* __restrict__ z, int B, int Hz, int Wz, const float* __restrict__ bias, int act, int crop,
                  float* __restrict__ out, int tiles_x, int tiles_y) {
  extern __shared__ uint32_t tg_sm[];
  constexpr int PH = TG_H + KH - 1, PW = TG_W + KW - 1;
  constexpr int ZW = sizeof(T) == 2 ? ZC / 2 : ZC;        // 32-bit words per pixel
  constexpr int PITCH = ZW + 1;
  const int Ho = Hz - KH + 1 - 2 * crop, Wo = Wz - KW + 1 - 2 * crop;
  int tix = blockIdx.x;
  const int tx0 = (tix % tiles_x) * TG_W; tix /= tiles_x;
  const int ty0 = (tix % tiles_y) * TG_H;
  const int n = tix / tiles_y;
  // staging: one thread copies one 16-byte chunk (CH chunks per pixel); 4 independent loads in flight per thread
  constexpr int CH = (ZC * (int)sizeof(T)) / 16;             // 16-byte chunks per pixel (8 on the 16-bit paths)
  constexpr int ITEMS = PH * PW * CH;
  for (int i0 = threadIdx.x; i0 < ITEMS; i0 += 256 * 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 256;
      v[u] = make_uint4(0u, 0u, 0u, 0u);
      if (i < ITEMS) {
        const int pix = i / CH, c = i - pix * CH;
        const int py = pix / PW, px = pix - py * PW;
        const int gy = ty0 + crop + py, gx = tx0 + crop + px;
        if (gy < Hz && gx < Wz)
          v[u] = ldg_stream16(reinterpret_cast<const uint8_t*>(z + (((size_t)n * Hz + gy) * Wz + gx) * ZC) + c * 16);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 256;
      if (i < ITEMS) {
        const int pix = i / CH, c = i - pix * CH;
        uint32_t* d = tg_sm + pix * PITCH + c * 4;           // odd pitch: four 4-byte stores
        d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w;
      }
    }
  }
  __syncthreads();
  const int lx = threadIdx.x % TG_W, ly = threadIdx.x / TG_W;
  const int ox = tx0 + lx, oy = ty0 + ly;
  if (ox >= Wo || oy >= Ho) return;
  float s = 0.f;
#pragma unroll
  for (int kh = 0; kh < KH; ++kh)
#pragma unroll
    for (int kw = 0; kw < KW; ++kw) {
      constexpr int dummy = 0; (void)dummy;
      const int t = kh * KW + kw;
      const int pix = (ly + kh) * PW + lx + kw;
      if constexpr (sizeof(T) == 2) {
        const float2 v = unpack2<T>(tg_sm[pix * PITCH + (t >> 1)]);
        s += (t & 1) ? v.y : v.x;
      } else {
        s += __uint_as_float(tg_sm[pix * PITCH + t]);
      }
    }
  out[((size_t)n * Ho + oy) * Wo + ox] = apply_act(s + (bias ? bias[0] : 0.f), act, 0.f);
}

static inline unsigned grid_for(long long work_items, int threads) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 8;   // 8 resident CTAs of 256 threads per SM
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

}  // namespace ng

using namespace ng;

#define DISPATCH_DTYPE(dtype, CALL)                                         \
  switch (dtype) {                                                          \
    case NG_F32: { using T = float; CALL; break; }                          \
    case NG_F16: { using T = __half; CALL; break; }                         \
    case NG_BF16: { using T = __nv_bfloat16; CALL; break; }                 \
    default: ng::set_error("bad dtype %d", (int)(dtype)); return NG_E_ARG;  \
  }

extern "C" int ng_pack_weight(const float* src, int32_t d0, int32_t d1, int32_t KH, int32_t KW, int32_t n_axis,
                              int32_t n_pad, int32_t k_pad, int32_t dtype, void* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src && dst && (n_axis == 0 || n_axis == 1), NG_E_ARG, "pack_weight: bad arguments");
  const int nn = n_axis == 0 ? d0 : d1, kk = n_axis == 0 ? d1 : d0;
  NG_REQUIRE(n_pad >= nn && k_pad >= kk, NG_E_SHAPE, "pack_weight: padding smaller than the tensor");
  const long long total = (long long)KH * KW * n_pad * k_pad;
  DISPATCH_DTYPE(dtype, (pack_weight_kernel<T><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
                            src, d0, d1, KH * KW, n_axis, n_pad, k_pad, (T*)dst)));
  NG_LAUNCH_CHECK("pack_weight_kernel");
  return NG_OK;
}

extern "C" int ng_pack_weight_phasemerged(const float* src, int32_t Cin, int32_t Cout, int32_t dtype, void* dst,
                                          void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src && dst && Cin > 0 && Cout > 0, NG_E_ARG, "pack_weight_phasemerged: bad arguments");
  DISPATCH_DTYPE(dtype, (pack_phasemerged_kernel<T><<<grid_for(16ll * Cout * Cin, 256), 256, 0, (cudaStream_t)stream>>>(
                            src, Cin, Cout, (T*)dst)));
  NG_LAUNCH_CHECK("pack_phasemerged_kernel");
  return NG_OK;
}

extern "C" int ng_unpack_weight_grad(const float* packed, int32_t d0, int32_t d1, int32_t KH, int32_t KW,
                                     int32_t n_axis, int32_t n_pad, int32_t k_pad, float scale,
                                     const float* dev_scale, float beta, float* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(packed && dst && (n_axis == 0 || n_axis == 1), NG_E_ARG, "unpack_weight_grad: bad arguments");
  const long long total = (long long)d0 * d1 * KH * KW;
  unpack_wgrad_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(packed, d0, d1, KH * KW, n_axis, n_pad,
                                                                             k_pad, scale, dev_scale, beta, dst);
  NG_LAUNCH_CHECK("unpack_wgrad_kernel");
  return NG_OK;
}

extern "C" int ng_prep_input(const float* src_a, int32_t ca, const float* src_b, int32_t cb, int32_t B, int32_t H,
                             int32_t W, int32_t wrap_pad, int32_t halo, int32_t halo_mode, int32_t c_pad,
                             int32_t dtype, void* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src_a && dst && ca > 0 && cb >= 0 && (cb == 0 || src_b), NG_E_ARG, "prep_input: bad arguments");
  NG_REQUIRE(c_pad >= ca + cb, NG_E_SHAPE, "prep_input: c_pad %d < %d channels", c_pad, ca + cb);
  NG_REQUIRE(wrap_pad < H && wrap_pad < W, NG_E_SHAPE, "prep_input: reflect pad %d needs a larger tile", wrap_pad);
  NG_REQUIRE(halo_mode != NG_HALO_REFLECT || (halo < H + 2 * wrap_pad && halo < W + 2 * wrap_pad), NG_E_SHAPE,
             "prep_input: halo too large");
  const long long total = (long long)B * (H + 2 * wrap_pad + 2 * halo) * (W + 2 * wrap_pad + 2 * halo);
  DISPATCH_DTYPE(dtype, (prep_input_kernel<T><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
                            src_a, ca, src_b, cb, B, H, W, wrap_pad, halo, halo_mode, c_pad, (T*)dst)));
  NG_LAUNCH_CHECK("prep_input_kernel");
  return NG_OK;
}

extern "C" int ng_prep_input_s2d(const float* src_a, int32_t ca, const float* src_b, int32_t cb, int32_t B, int32_t H,
                                 int32_t W, int32_t dtype, void* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src_a && dst && ca > 0 && cb >= 0 && (cb == 0 || src_b) && ca + cb <= 16, NG_E_ARG,
             "prep_input_s2d: bad arguments (at most 16 channels)");
  NG_REQUIRE(H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && dtype != NG_F32, NG_E_SHAPE,
             "prep_input_s2d: even H, W and 16-bit storage");
  const long long total = (long long)B * ((H + 2) / 2) * ((W + 2) / 2) * 4;
  if (dtype == NG_F16)
    prep_input_s2d_kernel<__half><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src_a, ca, src_b, cb, B, H, W, (__half*)dst);
  else
    prep_input_s2d_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src_a, ca, src_b, cb, B, H, W,
                                                                                               (__nv_bfloat16*)dst);
  NG_LAUNCH_CHECK("prep_input_s2d_kernel");
  return NG_OK;
}

extern "C" int ng_pack_weight_s2d(const float* src, int32_t O, int32_t I, int32_t transpose, int32_t dtype, void* dst,
                                  void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src && dst && O > 0 && I > 0 && I <= 16 && (transpose == 0 || transpose == 1), NG_E_ARG,
             "pack_weight_s2d: bad arguments");
  DISPATCH_DTYPE(dtype, (pack_weight_s2d_kernel<T><<<grid_for(4ll * O * 64, 256), 256, 0, (cudaStream_t)stream>>>(
                            src, O, I, transpose, (T*)dst)));
  NG_LAUNCH_CHECK("pack_weight_s2d_kernel");
  return NG_OK;
}

extern "C" int ng_unpack_weight_grad_s2d(const float* packed, int32_t O, int32_t I, float scale, const float* dev_scale,
                                         float beta, float* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(packed && dst && O > 0 && I > 0 && I <= 16, NG_E_ARG, "unpack_weight_grad_s2d: bad arguments");
  unpack_wgrad_s2d_kernel<<<grid_for((long long)O * I * 16, 256), 256, 0, (cudaStream_t)stream>>>(packed, O, I, scale,
                                                                                                   dev_scale, beta, dst);
  NG_LAUNCH_CHECK("unpack_wgrad_s2d_kernel");
  return NG_OK;
}

extern "C" int ng_in_stats(const void* y, int32_t dtype, int32_t B, int32_t HW, int32_t C, float* mean_rstd,
                           void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(y && mean_rstd && B > 0 && HW > 0 && C > 0, NG_E_ARG, "in_stats: bad arguments");
  dim3 grid(B, (C + 31) / 32);
  DISPATCH_DTYPE(dtype, (in_stats_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)y, HW, C, mean_rstd)));
  NG_LAUNCH_CHECK("in_stats_kernel");
  return NG_OK;
}

extern "C" int ng_in_stats_finalize(const float* partials, int32_t B, int32_t slots, int32_t C, int32_t count,
                                    float* mean_rstd, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(partials && mean_rstd && B > 0 && slots > 0 && C > 0 && count > 0, NG_E_ARG,
             "in_stats_finalize: bad arguments");
  NG_REQUIRE(C % 2 == 0, NG_E_SHAPE, "in_stats_finalize: C must be even");
  in_stats_finalize_kernel<<<(B * (C / 2) * 32 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      partials, B, slots, C, 1.0f / (float)count, mean_rstd);
  NG_LAUNCH_CHECK("in_stats_finalize_kernel");
  return NG_OK;
}

extern "C" int ng_memset_zero(void* ptr, int64_t bytes, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(ptr && bytes >= 0, NG_E_ARG, "memset_zero: bad arguments");
  return check_cuda(cudaMemsetAsync(ptr, 0, (size_t)bytes, (cudaStream_t)stream), "memset_zero");
}

extern "C" int ng_in_apply(const void* y, int32_t dtype, int32_t B, int32_t H, int32_t W, int32_t C,
                           const float* mean_rstd, const int64_t* stat_acc, float* mean_rstd_out, int32_t act,
                           float slope, const void* residual, int32_t res_pad,
                           const float* inject_e, int32_t inject_mode, const float* inject_scale, void* out,
                           int32_t out_pad, int32_t halo_mode, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(y && out, NG_E_ARG, "in_apply: null tensor");
  NG_REQUIRE(!(mean_rstd && stat_acc), NG_E_ARG, "in_apply: give mean_rstd or stat_acc, not both");
  NG_REQUIRE(((uintptr_t)stat_acc & 15) == 0 && ((uintptr_t)mean_rstd_out & 15) == 0, NG_E_ALIGN,
             "in_apply: statistics must be 16-byte aligned");
  NG_REQUIRE(C % 8 == 0, NG_E_SHAPE, "in_apply: C %d must be a multiple of 8", C);
  NG_REQUIRE(inject_mode == NG_INJECT_NONE || inject_e, NG_E_ARG, "in_apply: injection without embedding map");
  NG_REQUIRE(inject_mode == NG_INJECT_NONE || inject_mode == NG_INJECT_MUL || inject_scale, NG_E_ARG,
             "in_apply: scaled injection without scale_param");
  NG_REQUIRE(halo_mode != NG_HALO_REFLECT || (out_pad < H && out_pad < W), NG_E_SHAPE, "in_apply: halo too large");
  NG_REQUIRE(((uintptr_t)y & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)residual & 15) == 0, NG_E_ALIGN,
             "in_apply: tensors must be 16-byte aligned");
  const int C8 = C / 8;
  NG_REQUIRE((C8 & (C8 - 1)) == 0, NG_E_SHAPE, "in_apply: C/8 must be a power of two (C = %d)", C);
  int c8_shift = 0;
  while ((1 << c8_shift) < C8) ++c8_shift;
  const int Ho = H + 2 * out_pad, Wo = W + 2 * out_pad;
  NG_REQUIRE((long long)Ho * Wo < (1ll << 20) && Wo < (1 << 12), NG_E_SHAPE, "in_apply: image %dx%d too large", Ho, Wo);
  const unsigned long long wo_magic = ((1ull << 40) + (unsigned)Wo - 1) / (unsigned)Wo;   // exact for p < 2^20
  const int pstep = 256 / C8;                     // pixels per block per load
  // 16 sixteen-byte items per thread = 4 batches of UNROLL 4.  Tuning the multiplier for the wave efficiency of the grid
  // (B = 32 ResnetBlock units: 1120 blocks = 2.52 waves at 3 blocks / SM -> 832 blocks = 1.87 waves) measured SLOWER
  // end to end (r2z: 7639 vs 7813 tiles/s): these kernels run beside the other slice's persistent convolution, not alone.
  const int mult = 16;
  const int ppb = pstep * mult;
  dim3 grid((unsigned)((Ho * Wo + ppb - 1) / ppb), (unsigned)B);
  static const int apply_pf = [] { const char* e = getenv("NIRGAN_B200_APPLY_PREFETCH"); return e ? atoi(e) : 1; }();
  // lean kernel for the common case (see in_apply_fast_kernel); NIRGAN_B200_APPLY_FAST=0 keeps the generic one
  static const bool fast_on = [] { const char* e = getenv("NIRGAN_B200_APPLY_FAST"); return !(e && e[0] == '0'); }();
  const bool has_inj0 = inject_mode != NG_INJECT_NONE;
  if (fast_on && dtype != NG_F32 && (!has_inj0 || residual == nullptr) && (mean_rstd || stat_acc) &&
      (act == NG_ACT_RELU || act == NG_ACT_NONE) &&
      (long long)(H + 2 * (residual ? res_pad : 0)) * (W + 2 * (residual ? res_pad : 0)) * C < (1ll << 31) &&
      (long long)Ho * Wo * C < (1ll << 31)) {              // 32-bit element offsets inside one image
    const int reflect = halo_mode == NG_HALO_REFLECT ? 1 : 0;
    // NIRGAN_B200_APPLY_VARIANT: 0 = four 16-byte items in flight per thread at 3 blocks / SM (default), 1 = eight at 2,
    // 2 = four at 4 (<= 64 registers), 3 = two at 4
    static const int variant = [] { const char* e = getenv("NIRGAN_B200_APPLY_VARIANT"); return e ? atoi(e) : 0; }();
#define NG_FAST_ARGS(TT)                                                                                             \
        (const TT*)y, H, W, C, c8_shift, mean_rstd, (const long long*)stat_acc, mean_rstd_out, (const TT*)residual,    \
        res_pad, (TT*)out, out_pad, reflect, ppb, apply_pf
#define NG_FAST(TT, RES, RL)                                                                                         \
    do {                                                                                                             \
      if (variant == 1) in_apply_fast_kernel<TT, 8, RES, RL, 2><<<grid, 256, 0, (cudaStream_t)stream>>>(NG_FAST_ARGS(TT));      \
      else if (variant == 2) in_apply_fast_kernel<TT, 4, RES, RL, 4><<<grid, 256, 0, (cudaStream_t)stream>>>(NG_FAST_ARGS(TT)); \
      else if (variant == 3) in_apply_fast_kernel<TT, 2, RES, RL, 4><<<grid, 256, 0, (cudaStream_t)stream>>>(NG_FAST_ARGS(TT)); \
      else in_apply_fast_kernel<TT, 4, RES, RL, 3><<<grid, 256, 0, (cudaStream_t)stream>>>(NG_FAST_ARGS(TT));                   \
    } while (0)
#define NG_FAST_INJ(TT, RL)                                                                                          \
    in_apply_fast_kernel<TT, 4, false, RL, 3, true><<<grid, 256, 0, (cudaStream_t)stream>>>(NG_FAST_ARGS(TT), inject_e,    \
                                                                                           inject_mode, inject_scale)
#define NG_FAST_T(TT)                                                                                                \
    do {                                                                                                             \
      if (has_inj0) { if (act == NG_ACT_RELU) NG_FAST_INJ(TT, true); else NG_FAST_INJ(TT, false); }                 \
      else if (residual) { if (act == NG_ACT_RELU) NG_FAST(TT, true, true); else NG_FAST(TT, true, false); }        \
      else { if (act == NG_ACT_RELU) NG_FAST(TT, false, true); else NG_FAST(TT, false, false); }                    \
    } while (0)
    if (dtype == NG_F16) NG_FAST_T(__half); else NG_FAST_T(__nv_bfloat16);
#undef NG_FAST_T
#undef NG_FAST_INJ
#undef NG_FAST
#undef NG_FAST_ARGS
    NG_LAUNCH_CHECK("in_apply_fast_kernel");
    return NG_OK;
  }
#define NG_APPLY_LAUNCH(RES, INJ)                                                                                  \
  DISPATCH_DTYPE(dtype, (in_apply_kernel<T, 4, RES, INJ><<<grid, 256, 0, (cudaStream_t)stream>>>(                  \
                            (const T*)y, H, W, C, c8_shift, mean_rstd, (const long long*)stat_acc, mean_rstd_out, act,    \
                            slope, (const T*)residual, res_pad,                                                     \
                            inject_e, inject_mode, inject_scale, (T*)out, out_pad, halo_mode, ppb, wo_magic, apply_pf)))
  const bool has_inj = inject_mode != NG_INJECT_NONE;
  if (residual && has_inj) { NG_APPLY_LAUNCH(true, true); }
  else if (residual) { NG_APPLY_LAUNCH(true, false); }
  else if (has_inj) { NG_APPLY_LAUNCH(false, true); }
  else { NG_APPLY_LAUNCH(false, false); }
#undef NG_APPLY_LAUNCH
  NG_LAUNCH_CHECK("in_apply_kernel");
  return NG_OK;
}

extern "C" int ng_linear(const float* x, const float* w, const float* bias, int32_t B, int32_t K, int32_t N,
                         float* y, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(x && w && y && B > 0 && K > 0 && N > 0, NG_E_ARG, "linear: bad arguments");
  dim3 grid((N + 63) / 64, (B + 63) / 64);
  linear_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, w, bias, B, K, N, y);
  NG_LAUNCH_CHECK("linear_kernel");
  return NG_OK;
}

// scratch for the two-stage reductions lives in caller memory for ng_rs_pixel_losses; lsgan maps are tiny
// (B*30*30) so a single block suffices and needs no scratch.
extern "C" int ng_lsgan_loss(const float* p, int64_t n, float target, float* loss, int32_t accumulate, float* grad,
                             float gscale, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(p && loss && n > 0, NG_E_ARG, "lsgan_loss: bad arguments");
  // single block: the PatchGAN map is B x 30 x 30; deterministic and scratch-free
  static_assert(sizeof(float) == 4, "");
  float* partial = loss + 1;   // loss must have room for 2 floats: [0] = loss, [1] = scratch
  lsgan_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(p, (long long)n, target, partial, grad,
                                                   gscale * 2.0f / (float)n);
  NG_LAUNCH_CHECK("lsgan_kernel");
  reduce_partials_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(partial, 1, 1, 1.0f / (float)n, loss, accumulate);
  NG_LAUNCH_CHECK("reduce_partials_kernel");
  return NG_OK;
}

extern "C" int ng_rs_pixel_losses(const float* rgb, const float* nir, const float* pred, int32_t B, int32_t HW,
                                  const float* weights7, const float* weights7_dev, int32_t criterion, int32_t mask,
                                  float* out7, float* dpred, float* scratch, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(rgb && nir && pred && out7 && scratch && (weights7 || weights7_dev), NG_E_ARG, "rs_pixel_losses: bad arguments");
  NG_REQUIRE((criterion == 0 || criterion == 1) && mask > 0 && mask < 128, NG_E_ARG, "rs_pixel_losses: bad criterion / mask");
  const long long total = (long long)B * HW;
  unsigned blocks = grid_for(total, 256);
  if (blocks > 1024) blocks = 1024;
  RsWeights wt;
  for (int k = 0; k < 7; ++k) wt.w[k] = weights7 ? weights7[k] : 0.f;
  rs_pixel_loss_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rgb, nir, pred, B, HW, wt, weights7_dev, criterion, mask,
                                                                1.0f / (float)total, scratch, dpred);
  NG_LAUNCH_CHECK("rs_pixel_loss_kernel");
  reduce_partials_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(scratch, (int)blocks, 8, 1.0f / (float)total, out7, 0);
  NG_LAUNCH_CHECK("reduce_partials_kernel");
  return NG_OK;
}

extern "C" int ng_rs_index(const float* rgb, const float* nir, const float* pred, int32_t B, int32_t HW, int32_t which,
                           int32_t loss_eps, float* out_target, float* out_pred, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(rgb && nir && pred && out_target && out_pred && which >= 1 && which <= 6, NG_E_ARG, "rs_index: bad arguments");
  rs_index_kernel<<<grid_for((long long)B * HW, 256), 256, 0, (cudaStream_t)stream>>>(rgb, nir, pred, B, HW, which,
                                                                                     loss_eps, out_target, out_pred);
  NG_LAUNCH_CHECK("rs_index_kernel");
  return NG_OK;
}

extern "C" int ng_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                            float beta2, float eps, int32_t step, float grad_scale, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(p && g && m && v && n > 0 && step >= 1, NG_E_ARG, "adam_step: bad arguments");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, (long long)n, lr, beta1, beta2, eps, bc1,
                                                                 sqrtf(bc2), grad_scale);
  NG_LAUNCH_CHECK("adam_kernel");
  return NG_OK;
}

extern "C" int ng_adam_multi(void* const* params_dev, const int64_t* offsets_dev, const int64_t* numel_dev,
                             int32_t ntensors, const float* g, float* m, float* v, int64_t total, float lr, float beta1, float beta2, float eps,
                             int32_t* step_counter_dev, float grad_scale, const int32_t* skip_flag, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(params_dev && offsets_dev && numel_dev && g && m && v && step_counter_dev && ntensors > 0 && total > 0, NG_E_ARG,
             "adam_multi: bad arguments");
  adam_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_counter_dev, skip_flag);
  NG_LAUNCH_CHECK("adam_advance_kernel");
  adam_multi_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float* const*>(params_dev), reinterpret_cast<const long long*>(offsets_dev),
      reinterpret_cast<const long long*>(numel_dev), ntensors, g, m, v,
      (long long)total, lr, beta1, beta2, eps, grad_scale, step_counter_dev, skip_flag);
  NG_LAUNCH_CHECK("adam_multi_kernel");
  return NG_OK;
}

extern "C" int ng_nonfinite_flag(const float* x, int64_t n, int32_t* flag, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(x && flag && n > 0, NG_E_ARG, "nonfinite_flag: bad arguments");
  int e = check_cuda(cudaMemsetAsync(flag, 0, sizeof(int32_t), (cudaStream_t)stream), "nonfinite_flag memset");
  if (e) return e;
  nonfinite_flag_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, (long long)n, flag);
  NG_LAUNCH_CHECK("nonfinite_flag_kernel");
  return NG_OK;
}

// 16-bit paths with at most 4 source channels (the RGB stem): the block first stages its source row -- both reflections
// resolved, converted once -- in shared memory, so that an item is three 16-bit shared loads and one 16-byte store instead
// of two reflections and three global loads (the kernel was instruction-bound: 62 % issue utilisation under ncu).
constexpr int PS_MAXW = 2048 + 8;
template <typename T>
__global__ void __launch_bounds__(256)
prep_stem_smem_kernel(const float* __restrict__ src, int cin, int B, int H, int W, int wrap, int halo, int KW,
                      T* __restrict__ dst) {
  __shared__ uint16_t srow_s[4][PS_MAXW];
  const int H1 = H + 2 * wrap, W1 = W + 2 * wrap, Hb = H1 + 2 * halo;
  const int row = blockIdx.x;
  const int yb = row % Hb, n = row / Hb;
  const int y0 = reflect_idx(reflect_idx(yb - halo, H1) - wrap, H);
  const float* srow = src + ((size_t)n * cin * H + y0) * W;
  const size_t plane = (size_t)H * W;
  const int Wp = W1 + 8;                                  // x + kw for x < W1, kw < 8
  for (int j = threadIdx.x; j < Wp; j += 256) {
    const int x0 = reflect_idx(reflect_idx(min(j - halo, W1 - 1 + halo), W1) - wrap, W);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const T v = from_f32<T>(c < cin ? srow[c * plane + x0] : 0.f);
      srow_s[c][j] = *reinterpret_cast<const uint16_t*>(&v);
    }
  }
  __syncthreads();
  uint4* drow = reinterpret_cast<uint4*>(dst + (size_t)row * W1 * 64);
  for (int i = threadIdx.x; i < W1 * 8; i += 256) {
    const int kw = i & 7, x = i >> 3;
    uint4 u = make_uint4(0u, 0u, 0u, 0u);
    if (kw < KW) {
      const int j = x + kw;
      u.x = (uint32_t)srow_s[0][j] | ((uint32_t)srow_s[1][j] << 16);
      u.y = (uint32_t)srow_s[2][j] | ((uint32_t)srow_s[3][j] << 16);
    }
    drow[i] = u;
  }
}

extern "C" int ng_prep_stem(const float* src, int32_t cin, int32_t B, int32_t H, int32_t W, int32_t wrap_pad,
                            int32_t halo, int32_t KW, int32_t dtype, void* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src && dst && cin > 0 && cin <= 8 && KW > 0 && KW <= 8, NG_E_ARG, "prep_stem: cin and KW must be in 1..8");
  NG_REQUIRE(wrap_pad < H && wrap_pad < W && halo < H + 2 * wrap_pad && halo < W + 2 * wrap_pad, NG_E_SHAPE,
             "prep_stem: reflect padding needs a larger tile");
  const long long rows = (long long)B * (H + 2 * wrap_pad + 2 * halo);
  NG_REQUIRE(rows < (1ll << 31), NG_E_SHAPE, "prep_stem: too many rows");
  if (dtype != NG_F32 && cin <= 4 && W + 2 * wrap_pad + 8 <= PS_MAXW) {
    if (dtype == NG_F16)
      prep_stem_smem_kernel<__half><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(src, cin, B, H, W, wrap_pad, halo, KW,
                                                                                     (__half*)dst);
    else
      prep_stem_smem_kernel<__nv_bfloat16><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(src, cin, B, H, W, wrap_pad,
                                                                                            halo, KW, (__nv_bfloat16*)dst);
    NG_LAUNCH_CHECK("prep_stem_smem_kernel");
    return NG_OK;
  }
  DISPATCH_DTYPE(dtype, (prep_stem_kernel<T><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(
                            src, cin, B, H, W, wrap_pad, halo, KW, (T*)dst)));
  NG_LAUNCH_CHECK("prep_stem_kernel");
  return NG_OK;
}

extern "C" int ng_pack_weight_rowmerged(const float* src, int32_t O, int32_t I, int32_t KH, int32_t KW, int32_t c_slots,
                                        int32_t dtype, void* dst, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(src && dst && (c_slots == 8 || c_slots == 4) && I > 0 && I <= c_slots && KW > 0 && KW <= 8, NG_E_ARG,
             "pack_weight_rowmerged: c_slots 4 or 8, I <= c_slots, KW in 1..8");
  DISPATCH_DTYPE(dtype, (pack_rowmerged_kernel<T><<<grid_for((long long)KH * O * 8 * c_slots, 256), 256, 0, (cudaStream_t)stream>>>(
                            src, O, I, KH, KW, c_slots, (T*)dst)));
  NG_LAUNCH_CHECK("pack_rowmerged_kernel");
  return NG_OK;
}

extern "C" int ng_unpack_weight_grad_rowmerged(const float* packed, int32_t O, int32_t I, int32_t KH, int32_t KW,
                                               float scale, const float* dev_scale, float beta, float* dst,
                                               void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(packed && dst && I > 0 && I <= 8 && KW > 0 && KW <= 8, NG_E_ARG, "unpack_weight_grad_rowmerged: bad arguments");
  unpack_rowmerged_kernel<<<grid_for((long long)O * I * KH * KW, 256), 256, 0, (cudaStream_t)stream>>>(packed, O, I, KH,
                                                                                                      KW, scale, dev_scale, beta, dst);
  NG_LAUNCH_CHECK("unpack_rowmerged_kernel");
  return NG_OK;
}

extern "C" int ng_tap_gather(const void* z, int32_t dtype, int32_t B, int32_t Hz, int32_t Wz, int32_t zc, int32_t KH,
                             int32_t KW, const float* bias, int32_t act, int32_t crop, float* out, void* stream) {
  int r = require_sm100(); if (r) return r;
  NG_REQUIRE(z && out && KH * KW <= zc, NG_E_ARG, "tap_gather: need KH*KW <= zc");
  NG_REQUIRE(Hz - KH + 1 - 2 * crop > 0 && Wz - KW + 1 - 2 * crop > 0, NG_E_SHAPE, "tap_gather: empty output");
  NG_REQUIRE(KH == 7 && KW == 7 && zc == 64, NG_E_UNSUPPORTED, "tap_gather: built for 7x7 taps over 64 stored channels");
  const int Ho = Hz - KH + 1 - 2 * crop, Wo = Wz - KW + 1 - 2 * crop;
  const int tiles_x = (Wo + TG_W - 1) / TG_W, tiles_y = (Ho + TG_H - 1) / TG_H;
  const int row_words = dtype == NG_F32 ? zc : zc / 2;
  const size_t smem = (size_t)(TG_H + KH - 1) * (TG_W + KW - 1) * (row_words + 1) * 4;
  {
    cudaError_t e1 = cudaSuccess;
    switch (dtype) {
      case NG_F32: e1 = cudaFuncSetAttribute(tap_gather_kernel<float, 7, 7, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); break;
      case NG_F16: e1 = cudaFuncSetAttribute(tap_gather_kernel<__half, 7, 7, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); break;
      case NG_BF16: e1 = cudaFuncSetAttribute(tap_gather_kernel<__nv_bfloat16, 7, 7, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); break;
    }
    int e = check_cuda(e1, "tap_gather smem attribute");
    if (e) return e;
  }
  DISPATCH_DTYPE(dtype, (tap_gather_kernel<T, 7, 7, 64><<<(unsigned)((long long)B * tiles_x * tiles_y), 256, smem, (cudaStream_t)stream>>>(
                            (const T*)z, B, Hz, Wz, bias, act, crop, out, tiles_x, tiles_y)));
  NG_LAUNCH_CHECK("tap_gather_kernel");
  return NG_OK;
}
